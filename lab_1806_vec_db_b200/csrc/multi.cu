// multi.cu — the row-sharded search behind the C ABI: ONE process, one worker thread + stream per shard, results
// merged over NVLink peer memory (no NCCL, no host round trips between the phases).
//
// The reference's seam is one `knn` call on one index (src/index_algorithm/mod.rs:84-91), whatever hardware serves
// it; a Rust host therefore calls vdb_flat_knn once and this file spreads the call over the devices registered with
// vdb_init (SURVEY.md section 8e: contiguous row blocks per GPU, queries replicated, per-GPU top-k merged by
// (distance, global id) — contiguous blocks keep "lower id wins ties" identical to the unsharded scan).
//
// Per call, shard s (worker thread s, device dev[s], stream st[s]) runs
//   P0  (host queries) H2D of ITS 1/G slice of the batch over its own PCIe link, then peer stores of that slice into
//       every other shard's query buffer (NVLink) — instead of pushing the whole batch through every link
//   P1  tensor path: begin + SAMPLE -> its [nq, j] smallest sampled pruning scores, peer-stored into every shard's
//       gather buffer (the thresholds must be GLOBAL, or every shard reranks its own ~k candidates per query)
//   P2  TAU (merge of the G sample lists) -> FILTER + exact rerank -> its [nq, k] keys + per-query overflow flags;
//       the rows of the queries OWNED by shard h (a 1/G slice of the batch) are peer-stored straight into h's merge
//       buffer  (scan path: P1/P2 are one exact streaming scan)
//   P3  every shard merges the G lists of the nq/G queries it owns, runs the completeness check on them and writes
//       its slice of the result (host call: D2H over its own PCIe link)
// Between the phases the shards synchronise on the DEVICE (cudaStreamWaitEvent on the peers' events); the worker
// threads only meet at a spin barrier so that an event is recorded before a peer waits on it. The host reads one
// word per shard at the end (number of queries whose result could not be proven complete: 0 on the bench workload);
// flagged queries are re-run by the exact scan on every shard and merged on shard 0.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstring>
#include <functional>
#include <mutex>
#include <thread>
#include <vector>

#include "dataset.cuh"
#include "index.cuh"
#include "topk.cuh"

namespace vdb {

// ---- device list (vdb_init) ----------------------------------------------------------------------------------
static std::mutex g_init_mu;
static std::vector<int> g_devices;   // empty / one entry: single-device mode

std::vector<int> registered_devices() {
    std::lock_guard<std::mutex> lk(g_init_mu);
    return g_devices;
}

static void enable_peers(const std::vector<int>& devs) {
    int prev = 0;
    VDB_CUDA(cudaGetDevice(&prev));
    for (int a : devs)
        for (int b : devs) {
            if (a == b) continue;
            int can = 0;
            VDB_CUDA(cudaDeviceCanAccessPeer(&can, a, b));
            VDB_REQUIRE(can, "device %d cannot access device %d (no P2P path): the sharded search needs peer memory", a, b);
            VDB_CUDA(cudaSetDevice(a));
            cudaError_t e = cudaDeviceEnablePeerAccess(b, 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
            else VDB_CUDA(e);
        }
    VDB_CUDA(cudaSetDevice(prev));
}

// peer access between the listed devices; `register_default`: vdb_dataset_create shards over them from now on
void init_devices(const int* devices, uint32_t n, bool register_default) {
    std::vector<int> devs(devices, devices + n);
    int have = 0;
    VDB_CUDA(cudaGetDeviceCount(&have));
    for (int d : devs) VDB_REQUIRE(d >= 0 && d < have, "device %d out of range (have %d)", d, have);
    VDB_REQUIRE(n <= 64, "at most 64 shards");
    enable_peers(devs);
    if (!register_default) return;
    std::lock_guard<std::mutex> lk(g_init_mu);
    g_devices = devs;
}

// ---- small kernels ---------------------------------------------------------------------------------------------
constexpr int MAX_SHARDS = 64;
struct PtrList {
    void* p[MAX_SHARDS];
};

// src (16-byte aligned, n16 uint4) -> every dst[i], i < ndst (peer memory: 128-bit stores over NVLink)
__global__ void __launch_bounds__(256) bcast_kernel(const uint4* __restrict__ src, uint64_t n16, PtrList dst, uint32_t ndst) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint4 v = src[i];
        for (uint32_t d = 0; d < ndst; ++d) reinterpret_cast<uint4*>(dst.p[d])[i] = v;
    }
}

// rows of the queries owned by shard h go to h's merge buffer: keys [nq][k] -> dst_keys[h] + (q - lo_h) * k,
// flags [nq] -> dst_flags[h] + (q - lo_h). Owner of q = q / per.
__global__ void __launch_bounds__(128) scatter_owner_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ flags,
                                                           uint32_t nq, uint32_t k, uint32_t per, PtrList dst_keys,
                                                           PtrList dst_flags) {
    const uint32_t q = blockIdx.x;
    if (q >= nq) return;
    const uint32_t h = q / per, r = q - h * per;
    uint64_t* out = reinterpret_cast<uint64_t*>(dst_keys.p[h]) + (size_t)r * k;
    for (uint32_t j = threadIdx.x; j < k; j += blockDim.x) out[j] = keys[(size_t)q * k + j];
    if (flags && threadIdx.x == 0) reinterpret_cast<uint32_t*>(dst_flags.p[h])[r] = flags[q];
}

__global__ void or_flags_kernel(const uint32_t* __restrict__ in, uint32_t nlists, uint32_t cnt, uint32_t* __restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= cnt) return;
    uint32_t v = 0;
    for (uint32_t l = 0; l < nlists; ++l) v |= in[(size_t)l * cnt + i];
    out[i] = v;
}

__global__ void gather_query_rows_kernel(const uint8_t* __restrict__ src, uint32_t row_bytes, const uint32_t* __restrict__ idx,
                                         uint32_t cnt, uint8_t* __restrict__ dst) {
    const uint32_t i = blockIdx.x;
    if (i >= cnt) return;
    for (uint32_t e = threadIdx.x; e < row_bytes; e += blockDim.x)
        dst[(size_t)i * row_bytes + e] = src[(size_t)idx[i] * row_bytes + e];
}

// ---- worker pool -----------------------------------------------------------------------------------------------
// sense-reversing spin barrier of the shard workers (they are all running when they meet here)
struct SpinBarrier {
    std::atomic<uint32_t> count{0};
    std::atomic<uint32_t> sense{0};
    uint32_t n = 1;
    void wait() {
        const uint32_t s = sense.load(std::memory_order_acquire);
        if (count.fetch_add(1, std::memory_order_acq_rel) + 1 == n) {
            count.store(0, std::memory_order_relaxed);
            sense.store(s + 1, std::memory_order_release);
        } else {
            uint32_t spins = 0;
            while (sense.load(std::memory_order_acquire) == s)
                if (++spins > 4096) std::this_thread::yield();
        }
    }
};

// grow-only device buffer allocated with cudaMalloc (peer-accessible once peer access is enabled)
struct PeerBuf {
    void* p = nullptr;
    size_t cap = 0;
    void ensure(size_t bytes) {   // current device = the owning shard's
        if (bytes <= cap) return;
        if (p) VDB_CUDA(cudaFree(p));
        p = nullptr;
        cap = 0;
        const size_t want = std::max<size_t>(bytes + bytes / 4, 4096);
        VDB_CUDA(cudaMalloc(&p, want));
        cap = want;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

enum { EV_Q = 0, EV_S, EV_P, EV_F, EV_R, EV_COUNT };

struct Shard {
    int device = 0;
    vdb_dataset* ds = nullptr;
    uint64_t lo = 0, hi = 0;          // global row block
    cudaStream_t st = nullptr;
    cudaEvent_t ev[EV_COUNT] = {};
    PeerBuf q_all, jall, ustat, kin, ovin;   // written by the peers
    PeerBuf out_ids, out_dist, out_cnt;   // host calls: this shard's slice of the result before the D2H
    uint32_t* h_redo = nullptr;       // pinned: [0] = count, [1..] = flagged batch indices of the owned slice
    size_t h_redo_cap = 0;
    uint64_t* h_stat = nullptr;       // pinned: candidates reranked by this shard in the call
    std::thread th;
};

}  // namespace vdb

struct vdb_sharded_state {
    std::vector<vdb::Shard> shards;
    // job hand-off
    std::mutex mu;
    std::condition_variable cv_work, cv_done;
    std::atomic<uint64_t> gen{0};
    std::atomic<uint32_t> done{0};
    std::atomic<uint32_t> sleepers{0};
    bool stop = false;
    const std::vector<std::function<void(uint32_t)>>* phases = nullptr;
    std::atomic<bool> failed{false};
    std::mutex err_mu;
    std::string err;
    int err_code = VDB_ECUDA;
    vdb::SpinBarrier barrier;
    std::mutex call_mu;               // one sharded call at a time (every GPU is busy with it anyway)
    // tensor-path facts, gathered on first use
    bool tensor_known = false, tensor_ok = false;
    uint64_t ns_total = 0, ns_min = 0;
    float mean_norm = 0.f, mean_ex = 0.f;
};

namespace vdb {

static void worker_main(vdb_sharded_state* S, uint32_t s) {
    cudaSetDevice(S->shards[s].device);
    uint64_t seen = 0;
    for (;;) {
        // wait for the next job: spin briefly (back-to-back calls), then sleep
        uint32_t spins = 0;
        while (S->gen.load(std::memory_order_acquire) == seen) {
            if (++spins < 20000) continue;
            std::unique_lock<std::mutex> lk(S->mu);
            S->sleepers.fetch_add(1);
            S->cv_work.wait(lk, [&] { return S->stop || S->gen.load(std::memory_order_acquire) != seen; });
            S->sleepers.fetch_sub(1);
            break;
        }
        {
            std::lock_guard<std::mutex> lk(S->mu);
            if (S->stop) return;
        }
        seen = S->gen.load(std::memory_order_acquire);
        const auto& phases = *S->phases;
        static const bool trace = getenv("VDB_MG_TRACE") != nullptr;   // host time each phase takes to enqueue (diagnostic)
        double host_us[8] = {};
        for (size_t p = 0; p < phases.size(); ++p) {
            const auto t0 = std::chrono::steady_clock::now();
            if (!S->failed.load(std::memory_order_acquire)) {
                try {
                    phases[p](s);
                } catch (const Error& e) {
                    std::lock_guard<std::mutex> lk(S->err_mu);
                    if (!S->failed.exchange(true)) S->err = e.what(), S->err_code = e.code;
                } catch (const std::exception& e) {
                    std::lock_guard<std::mutex> lk(S->err_mu);
                    if (!S->failed.exchange(true)) S->err = e.what(), S->err_code = VDB_ECUDA;
                }
            }
            if (trace && p < 8) host_us[p] = std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t0).count();
            if (p + 1 < phases.size()) S->barrier.wait();
        }
        if (trace && s == 0)
            fprintf(stderr, "[vdb mg] shard 0 host us per phase: %.0f %.0f %.0f %.0f %.0f\n", host_us[0], host_us[1], host_us[2], host_us[3],
                    host_us[4]);
        if (S->failed.load()) cudaStreamSynchronize(S->shards[s].st);   // nothing of the call may outlive it
        if (S->done.fetch_add(1, std::memory_order_acq_rel) + 1 == S->shards.size()) {
            std::lock_guard<std::mutex> lk(S->mu);
            S->cv_done.notify_all();
        }
    }
}

// runs the phases on every shard's worker thread; phases are separated by barriers; throws the first error
static void run_job(vdb_sharded_state* S, const std::vector<std::function<void(uint32_t)>>& phases) {
    S->phases = &phases;
    S->failed.store(false);
    S->done.store(0);
    S->gen.fetch_add(1, std::memory_order_release);
    if (S->sleepers.load() > 0) {
        std::lock_guard<std::mutex> lk(S->mu);
        S->cv_work.notify_all();
    }
    const uint32_t G = (uint32_t)S->shards.size();
    uint32_t spins = 0;
    while (S->done.load(std::memory_order_acquire) != G) {
        if (++spins < 2000) continue;
        std::unique_lock<std::mutex> lk(S->mu);
        S->cv_done.wait_for(lk, std::chrono::microseconds(200), [&] { return S->done.load(std::memory_order_acquire) == G; });
    }
    S->phases = nullptr;
    if (S->failed.load()) throw Error(S->err_code, S->err);
}

static void wait_peers(vdb_sharded_state* S, uint32_t s, int ev) {
    for (uint32_t h = 0; h < S->shards.size(); ++h)
        if (h != s) VDB_CUDA(cudaStreamWaitEvent(S->shards[s].st, S->shards[h].ev[ev], 0));
}

static void bcast(const void* src, size_t bytes, const PtrList& dst, uint32_t ndst, cudaStream_t st) {
    if (bytes == 0 || ndst == 0) return;
    bool aligned = (((uintptr_t)src | bytes) & 15) == 0;
    for (uint32_t d = 0; d < ndst; ++d) aligned = aligned && (((uintptr_t)dst.p[d]) & 15) == 0;
    if (aligned) {
        const uint64_t n16 = bytes / 16;
        const uint32_t grid = (uint32_t)std::min<uint64_t>(ceil_div<uint64_t>(n16, 256), 4 * (uint64_t)sm_count());
        bcast_kernel<<<grid, 256, 0, st>>>((const uint4*)src, n16, dst, ndst);
        VDB_LAUNCHED();
    } else {
        for (uint32_t d = 0; d < ndst; ++d) VDB_CUDA(cudaMemcpyAsync(dst.p[d], src, bytes, cudaMemcpyDefault, st));
    }
}

// ---- create / destroy -------------------------------------------------------------------------------------------
void shard_bounds(uint64_t n, uint32_t world, uint32_t rank, uint64_t* lo, uint64_t* hi) {
    const uint64_t base = n / world, rem = n % world;
    *lo = rank * base + std::min<uint64_t>(rank, rem);
    *hi = *lo + base + (rank < rem ? 1 : 0);
}

void sharded_destroy(vdb_dataset* md) {
    vdb_sharded_state* S = md->sharded;
    if (S) {
        {
            std::lock_guard<std::mutex> lk(S->mu);
            S->stop = true;
            S->gen.fetch_add(1);
            S->cv_work.notify_all();
        }
        for (auto& sh : S->shards)
            if (sh.th.joinable()) sh.th.join();
        int prev = 0;
        cudaGetDevice(&prev);
        for (auto& sh : S->shards) {
            cudaSetDevice(sh.device);
            if (sh.st) cudaStreamSynchronize(sh.st);
            for (PeerBuf* b : {&sh.q_all, &sh.jall, &sh.ustat, &sh.kin, &sh.ovin, &sh.out_ids, &sh.out_dist, &sh.out_cnt}) b->release();
            if (sh.h_redo) cudaFreeHost(sh.h_redo);
            if (sh.h_stat) cudaFreeHost(sh.h_stat);
            for (auto& e : sh.ev)
                if (e) cudaEventDestroy(e);
            if (sh.st) cudaStreamDestroy(sh.st);
            if (sh.ds) vdb_dataset_destroy(sh.ds);
        }
        cudaSetDevice(prev);
        delete S;
    }
    delete md;
}

// shard datasets are created by `make_shard(s, device, lo, hi)` (upload of a host block / adoption of device rows)
vdb_dataset* sharded_create(const std::vector<int>& devs, uint64_t n, uint32_t dim, int dtype, int metric, uint64_t id_base,
                            const std::vector<uint64_t>* counts,
                            const std::function<vdb_dataset*(uint32_t, int, uint64_t, uint64_t)>& make_shard) {
    const uint32_t G = (uint32_t)devs.size();
    VDB_REQUIRE(G >= 1 && G <= MAX_SHARDS, "1..%d shards", MAX_SHARDS);
    auto md = new vdb_dataset();
    md->owned = false;
    md->n = md->cap = n;
    md->dim = dim;
    md->dtype = dtype;
    md->metric = metric;
    md->id_base = id_base;
    md->pitch = round_up(dim, vec_elems(dtype));
    md->device = devs[0];
    auto S = new vdb_sharded_state();
    md->sharded = S;
    S->shards.resize(G);
    S->barrier.n = G;
    int prev = 0;
    cudaGetDevice(&prev);
    try {
        uint64_t at = 0;
        for (uint32_t s = 0; s < G; ++s) {
            Shard& sh = S->shards[s];
            sh.device = devs[s];
            if (counts) {
                sh.lo = at;
                sh.hi = at + (*counts)[s];
                at = sh.hi;
            } else {
                shard_bounds(n, G, s, &sh.lo, &sh.hi);
            }
            VDB_CUDA(cudaSetDevice(sh.device));
            pool_init();
            VDB_CUDA(cudaStreamCreateWithFlags(&sh.st, cudaStreamNonBlocking));
            for (auto& e : sh.ev) VDB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            VDB_CUDA(cudaHostAlloc((void**)&sh.h_stat, 8, cudaHostAllocPortable));
            sh.ds = make_shard(s, sh.device, sh.lo, sh.hi);
        }
        VDB_CUDA(cudaSetDevice(prev));
        for (uint32_t s = 0; s < G; ++s) S->shards[s].th = std::thread(worker_main, S, s);
    } catch (...) {
        cudaSetDevice(prev);
        sharded_destroy(md);
        throw;
    }
    return md;
}

// ---- the sharded Flat search ---------------------------------------------------------------------------------------
constexpr uint32_t SHARD_TENSOR_MIN_NQ = 12;   // below: every shard runs the exact streaming scan (K1)
constexpr uint32_t SHARD_QUERY_CHUNK = 16384;  // bounds the candidate / rerank scratch of the filter phase

struct FlatCallArgs {
    const void* h_queries = nullptr;            // host call
    const void* const* d_queries = nullptr;     // device call: [G] replicated batches
    uint32_t nq = 0, k = 0;
    uint64_t* h_ids = nullptr;
    float* h_dist = nullptr;
    uint32_t* h_counts = nullptr;
    uint64_t* const* d_ids = nullptr;           // device call: [G] result slices on the owners
    float* const* d_dist = nullptr;
    uint32_t* const* d_counts = nullptr;
};

static void ensure_tensor_facts(const vdb_dataset* md) {
    vdb_sharded_state* S = md->sharded;
    if (S->tensor_known) return;
    const uint32_t G = (uint32_t)S->shards.size();
    std::vector<uint64_t> ns(G, 0);
    std::vector<float> mn(G, 0.f), me(G, 0.f);
    std::vector<int> ok(G, 0);
    std::vector<std::function<void(uint32_t)>> ph = {[&](uint32_t s) {
        Shard& sh = S->shards[s];
        if (!flat_gemm_supported(sh.ds, 1, 1)) return;
        uint64_t n = 0;
        uint32_t sn = 0;
        tensor_info(sh.ds, &n, &sn, &mn[s], &me[s], sh.st);
        VDB_CUDA(cudaStreamSynchronize(sh.st));
        ns[s] = sn;
        ok[s] = 1;
    }};
    run_job(S, ph);
    S->tensor_ok = true;
    S->ns_total = 0;
    S->ns_min = ~0ull;
    S->mean_norm = S->mean_ex = 0.f;
    for (uint32_t s = 0; s < G; ++s) {
        S->tensor_ok = S->tensor_ok && ok[s];
        S->ns_total += ns[s];
        S->ns_min = std::min<uint64_t>(S->ns_min, ns[s]);
        S->mean_norm = std::max(S->mean_norm, mn[s]);
        S->mean_ex = std::max(S->mean_ex, me[s]);
    }
    S->tensor_known = true;
}

// shard-local search of a single-exchange call (IVF): enqueues [nq, k] ascending keys for shard s on `st`
using KeyProducer = std::function<void(uint32_t s, const void* d_q, uint32_t nq, uint32_t k, uint64_t* d_keys, cudaStream_t st)>;

// one chunk of at most SHARD_QUERY_CHUNK queries. producer == nullptr: Flat (tensor phases or exact scan per shard)
static void sharded_flat_chunk(const vdb_dataset* md, const FlatCallArgs& a, int path, const KeyProducer* producer = nullptr) {
    vdb_sharded_state* S = md->sharded;
    const uint32_t G = (uint32_t)S->shards.size();
    const uint32_t nq = a.nq, k = a.k;
    const size_t rb = (size_t)md->dim * md->elem_size();
    const bool host = a.h_queries != nullptr;
    const uint32_t per = ceil_div(nq, G);
    auto slice = [&](uint32_t h, uint32_t* lo, uint32_t* hi) {
        *lo = std::min(nq, h * per);
        *hi = std::min(nq, (h + 1) * per);
    };
    bool tensor = false;
    if (!producer && path != 1 && k >= 1 && k <= 1024 && (path == 2 || nq >= SHARD_TENSOR_MIN_NQ)) {
        ensure_tensor_facts(md);
        tensor = S->tensor_ok;
        VDB_REQUIRE(tensor || path != 2, "tensor-core Flat path needs f32/u8 shards of at least 65536 rows and k <= 1024");
    }
    uint32_t j0 = 0, j = 0;
    if (tensor) {
        j0 = tensor_j0(k, S->ns_total, md->n);
        j = tensor_sample_j(j0, S->ns_min);
    }
    // small host batches are uploaded whole by every shard (no exchange); large ones slice by slice + NVLink broadcast
    const bool q_exchange = host && (size_t)nq * rb >= (256u << 10) && G > 1;

    // exchange buffers must exist before any peer writes into them
    {
        int prev = 0;
        VDB_CUDA(cudaGetDevice(&prev));
        for (uint32_t s = 0; s < G; ++s) {
            Shard& sh = S->shards[s];
            uint32_t lo, hi;
            slice(s, &lo, &hi);
            const uint32_t cnt = hi - lo;
            VDB_CUDA(cudaSetDevice(sh.device));
            if (host) sh.q_all.ensure((size_t)nq * rb);
            if (tensor) sh.jall.ensure((size_t)G * nq * j * 8);
            if (tensor) sh.ustat.ensure((size_t)G * nq * ((k + 3) / 4) * 4);   // global pruning statistics (GPRUNE_M = 4)
            sh.kin.ensure((size_t)G * std::max(cnt, 1u) * k * 8);
            sh.ovin.ensure((size_t)G * std::max(cnt, 1u) * 4);
            if (host) {
                sh.out_ids.ensure((size_t)std::max(cnt, 1u) * k * 8);
                sh.out_dist.ensure((size_t)std::max(cnt, 1u) * k * 4);
                sh.out_cnt.ensure((size_t)std::max(cnt, 1u) * 4);
            }
            const size_t need = (size_t)(cnt + 1) * 4;
            if (need > sh.h_redo_cap) {
                if (sh.h_redo) VDB_CUDA(cudaFreeHost(sh.h_redo));
                sh.h_redo = nullptr;
                VDB_CUDA(cudaHostAlloc((void**)&sh.h_redo, need * 2, cudaHostAllocPortable));
                sh.h_redo_cap = need * 2;
            }
            sh.h_redo[0] = 0;
            *sh.h_stat = 0;
        }
        VDB_CUDA(cudaSetDevice(prev));
    }

    std::vector<vdb_tq*> tqs(G, nullptr);
    std::vector<const void*> qptr(G, nullptr);
    struct Local {
        DevBuf jkeys, tau, keys, ovf, merged, ovm, redo, nredo;
    };
    std::vector<Local> loc(G);

    std::vector<std::function<void(uint32_t)>> ph;
    // P0: queries
    // vdb_prof_*: shard 0's device time per phase (a phase's span includes its wait for the slowest peer)
    struct PhaseProf {
        ProfScope* p = nullptr;
        PhaseProf(bool on, const char* name, cudaStream_t st) {
            if (on && g_prof_on) p = new ProfScope(name, st);
        }
        ~PhaseProf() { delete p; }
    };
    ph.push_back([&](uint32_t s) {
        Shard& sh = S->shards[s];
        PhaseProf pp(s == 0, "mg_queries", sh.st);
        if (!host) {
            qptr[s] = a.d_queries[s];
            return;
        }
        qptr[s] = sh.q_all.p;
        if (!q_exchange) {
            VDB_CUDA(cudaMemcpyAsync(sh.q_all.p, a.h_queries, (size_t)nq * rb, cudaMemcpyHostToDevice, sh.st));
            return;
        }
        uint32_t lo, hi;
        slice(s, &lo, &hi);
        if (hi > lo) {
            uint8_t* mine = (uint8_t*)sh.q_all.p + (size_t)lo * rb;
            VDB_CUDA(cudaMemcpyAsync(mine, (const uint8_t*)a.h_queries + (size_t)lo * rb, (size_t)(hi - lo) * rb,
                                     cudaMemcpyHostToDevice, sh.st));
            PtrList dst{};
            uint32_t nd = 0;
            for (uint32_t h = 0; h < G; ++h)
                if (h != s) dst.p[nd++] = (uint8_t*)S->shards[h].q_all.p + (size_t)lo * rb;
            bcast(mine, (size_t)(hi - lo) * rb, dst, nd, sh.st);
        }
        VDB_CUDA(cudaEventRecord(sh.ev[EV_Q], sh.st));
    });
    // P1: sample (tensor) / nothing (scan)
    ph.push_back([&](uint32_t s) {
        Shard& sh = S->shards[s];
        PhaseProf pp(s == 0, "mg_sample", sh.st);
        if (q_exchange) wait_peers(S, s, EV_Q);
        if (!tensor) return;
        tqs[s] = tensor_begin(sh.ds, qptr[s], nq, sh.st);
        loc[s].jkeys = DevBuf((size_t)nq * j * 8, sh.st);
        tensor_sample_keys(tqs[s], j, loc[s].jkeys.as<uint64_t>());
        PtrList dst{};
        for (uint32_t h = 0; h < G; ++h) dst.p[h] = (uint8_t*)S->shards[h].jall.p + (size_t)s * nq * j * 8;
        {
            PhaseProf pb(s == 0, "mg_bcast", sh.st);
            bcast(loc[s].jkeys.p, (size_t)nq * j * 8, dst, G, sh.st);
        }
        VDB_CUDA(cudaEventRecord(sh.ev[EV_S], sh.st));
    });
    // P2a (tensor path with the global pruning bound): thresholds + contraction + this shard's pruning statistics to every shard
    bool gprune = false;   // decided by shard 0 in P1 (same answer on every shard: it depends on k and the environment only)
    ph.push_back([&](uint32_t s) {
        if (!tensor || G < 2 || !tensor_filter_split_supported(tqs[s], k)) return;
        if (s == 0) gprune = true;
        Shard& sh = S->shards[s];
        Local& L = loc[s];
        PhaseProf pp(s == 0, "mg_filter", sh.st);
        wait_peers(S, s, EV_S);
        L.tau = DevBuf((size_t)nq * 4, sh.st);
        L.ovf = DevBuf((size_t)nq * 4, sh.st);
        tensor_tau(tqs[s], (const uint64_t*)sh.jall.p, G, j, (uint32_t)std::min<uint64_t>(j0, (uint64_t)j * G), L.tau.as<float>());
        uint32_t T = 0;
        const uint32_t* stats = tensor_filter_begin(tqs[s], k, L.tau.as<float>(), &T);
        PtrList dst{};
        for (uint32_t h = 0; h < G; ++h) dst.p[h] = (uint8_t*)S->shards[h].ustat.p + (size_t)s * nq * T * 4;
        bcast(stats, (size_t)nq * T * 4, dst, G, sh.st);
        VDB_CUDA(cudaEventRecord(sh.ev[EV_P], sh.st));
    });
    // P2: thresholds + filter + rerank (tensor) / exact scan; rows of the owned slices go to their owners
    ph.push_back([&](uint32_t s) {
        Shard& sh = S->shards[s];
        Local& L = loc[s];
        PhaseProf pp(s == 0, gprune ? "mg_finish" : "mg_filter", sh.st);
        L.keys = DevBuf((size_t)nq * k * 8, sh.st);
        if (tensor && gprune) {
            wait_peers(S, s, EV_P);
            tensor_filter_finish(tqs[s], (const uint32_t*)sh.ustat.p, G, L.keys.as<uint64_t>(), L.ovf.as<uint32_t>());
            VDB_CUDA(cudaMemcpyAsync(sh.h_stat, tensor_cand_total_ptr(tqs[s]), 8, cudaMemcpyDeviceToHost, sh.st));
        } else if (tensor) {
            wait_peers(S, s, EV_S);
            L.tau = DevBuf((size_t)nq * 4, sh.st);
            L.ovf = DevBuf((size_t)nq * 4, sh.st);
            tensor_tau(tqs[s], (const uint64_t*)sh.jall.p, G, j, (uint32_t)std::min<uint64_t>(j0, (uint64_t)j * G),
                       L.tau.as<float>());
            tensor_filter_keys(tqs[s], k, 0, L.tau.as<float>(), L.keys.as<uint64_t>(), L.ovf.as<uint32_t>());
            VDB_CUDA(cudaMemcpyAsync(sh.h_stat, tensor_cand_total_ptr(tqs[s]), 8, cudaMemcpyDeviceToHost, sh.st));
        } else if (producer) {
            (*producer)(s, qptr[s], nq, k, L.keys.as<uint64_t>(), sh.st);
        } else {
            flat_scan_keys(sh.ds, qptr[s], nq, k, L.keys.as<uint64_t>(), sh.st);
        }
        PtrList dk{}, df{};
        for (uint32_t h = 0; h < G; ++h) {
            uint32_t lo, hi;
            slice(h, &lo, &hi);
            const uint32_t cnt = std::max(hi - lo, 1u);
            dk.p[h] = (uint8_t*)S->shards[h].kin.p + (size_t)s * cnt * k * 8;
            df.p[h] = (uint8_t*)S->shards[h].ovin.p + (size_t)s * cnt * 4;
        }
        {
            PhaseProf ps(s == 0, "mg_scatter", sh.st);
            scatter_owner_kernel<<<nq, 128, 0, sh.st>>>(L.keys.as<uint64_t>(), tensor ? L.ovf.as<uint32_t>() : nullptr, nq, k, per,
                                                        dk, df);
            VDB_LAUNCHED();
        }
        VDB_CUDA(cudaEventRecord(sh.ev[EV_F], sh.st));
    });
    // P3: merge of the owned slice, completeness check, result slice
    ph.push_back([&](uint32_t s) {
        Shard& sh = S->shards[s];
        Local& L = loc[s];
        PhaseProf* pp = new PhaseProf(s == 0, "mg_merge", sh.st);
        wait_peers(S, s, EV_F);
        uint32_t lo, hi;
        slice(s, &lo, &hi);
        const uint32_t cnt = hi - lo;
        uint64_t* o_ids = host ? (uint64_t*)sh.out_ids.p : a.d_ids[s];
        float* o_dist = host ? (float*)sh.out_dist.p : a.d_dist[s];
        uint32_t* o_cnt = host ? (uint32_t*)sh.out_cnt.p : a.d_counts[s];
        if (cnt) {
            L.merged = DevBuf((size_t)cnt * k * 8, sh.st);
            launch_merge_sorted((const uint64_t*)sh.kin.p, G, cnt, k, k, L.merged.as<uint64_t>(), o_ids, o_dist, o_cnt, sh.st);
            if (tensor) {
                L.ovm = DevBuf((size_t)cnt * 4, sh.st);
                L.redo = DevBuf((size_t)cnt * 4, sh.st);
                L.nredo = DevBuf(4, sh.st);
                or_flags_kernel<<<ceil_div(cnt, 256u), 256, 0, sh.st>>>((const uint32_t*)sh.ovin.p, G, cnt, L.ovm.as<uint32_t>());
                VDB_LAUNCHED();
                tensor_check_range(tqs[s], lo, cnt, L.merged.as<uint64_t>(), k, md->n, L.tau.as<float>(), L.ovm.as<uint32_t>(),
                                   L.redo.as<uint32_t>(), L.nredo.as<uint32_t>());
                VDB_CUDA(cudaMemcpyAsync(sh.h_redo, L.nredo.p, 4, cudaMemcpyDeviceToHost, sh.st));
                VDB_CUDA(cudaMemcpyAsync(sh.h_redo + 1, L.redo.p, (size_t)cnt * 4, cudaMemcpyDeviceToHost, sh.st));
            }
            if (host) {
                VDB_CUDA(cudaMemcpyAsync(a.h_ids + (size_t)lo * k, o_ids, (size_t)cnt * k * 8, cudaMemcpyDeviceToHost, sh.st));
                VDB_CUDA(cudaMemcpyAsync(a.h_dist + (size_t)lo * k, o_dist, (size_t)cnt * k * 4, cudaMemcpyDeviceToHost, sh.st));
                VDB_CUDA(cudaMemcpyAsync(a.h_counts + lo, o_cnt, (size_t)cnt * 4, cudaMemcpyDeviceToHost, sh.st));
            }
        }
        L = Local();   // stream-ordered frees
        if (tqs[s]) tensor_end(tqs[s]), tqs[s] = nullptr;
        delete pp;
        VDB_CUDA(cudaStreamSynchronize(sh.st));
    });
    try {
        run_job(S, ph);
    } catch (...) {
        for (uint32_t s = 0; s < G; ++s)
            if (tqs[s]) {
                int prev = 0;
                cudaGetDevice(&prev);
                cudaSetDevice(S->shards[s].device);
                cudaStreamSynchronize(S->shards[s].st);
                loc[s] = Local();
                tensor_end(tqs[s]);
                cudaSetDevice(prev);
            }
        throw;
    }
    if (!tensor) return;

    // ---- flagged queries: exact scan on every shard, merged on shard 0 (rare: 0 of 240 000 on the bench workload) ----
    std::vector<uint32_t> redo;
    uint64_t cands = 0;
    for (uint32_t s = 0; s < G; ++s) {
        const Shard& sh = S->shards[s];
        cands += *sh.h_stat;
        for (uint32_t i = 0; i < sh.h_redo[0]; ++i) redo.push_back(sh.h_redo[1 + i]);
    }
    g_gemm_queries += nq;
    g_gemm_cands += cands;
    g_gemm_redo += redo.size();
    if (redo.empty()) return;
    std::sort(redo.begin(), redo.end());
    const uint32_t nr = (uint32_t)redo.size();
    std::vector<uint64_t> r_ids((size_t)nr * k);
    std::vector<float> r_dist((size_t)nr * k);
    std::vector<uint32_t> r_cnt(nr);
    {
        int prev = 0;
        VDB_CUDA(cudaGetDevice(&prev));
        VDB_CUDA(cudaSetDevice(S->shards[0].device));
        S->shards[0].kin.ensure((size_t)G * nr * k * 8);
        VDB_CUDA(cudaSetDevice(prev));
    }
    std::vector<std::function<void(uint32_t)>> rp;
    rp.push_back([&](uint32_t s) {
        Shard& sh = S->shards[s];
        DevBuf sel((size_t)nr * 4, sh.st), rq((size_t)nr * rb, sh.st), rk((size_t)nr * k * 8, sh.st);
        VDB_CUDA(cudaMemcpyAsync(sel.p, redo.data(), (size_t)nr * 4, cudaMemcpyHostToDevice, sh.st));
        gather_query_rows_kernel<<<nr, 128, 0, sh.st>>>((const uint8_t*)qptr[s], (uint32_t)rb, sel.as<uint32_t>(), nr, rq.as<uint8_t>());
        VDB_LAUNCHED();
        flat_scan_keys(sh.ds, rq.p, nr, k, rk.as<uint64_t>(), sh.st);
        VDB_CUDA(cudaMemcpyAsync((uint8_t*)S->shards[0].kin.p + (size_t)s * nr * k * 8, rk.p, (size_t)nr * k * 8,
                                 cudaMemcpyDefault, sh.st));
        VDB_CUDA(cudaEventRecord(sh.ev[EV_R], sh.st));
        if (s != 0) VDB_CUDA(cudaStreamSynchronize(sh.st));   // `redo` (host) and the scratch stay valid until here
    });
    rp.push_back([&](uint32_t s) {
        if (s != 0) return;
        Shard& sh = S->shards[0];
        wait_peers(S, 0, EV_R);
        DevBuf ids((size_t)nr * k * 8, sh.st), dd((size_t)nr * k * 4, sh.st), cn((size_t)nr * 4, sh.st);
        launch_merge_sorted((const uint64_t*)sh.kin.p, G, nr, k, k, nullptr, ids.as<uint64_t>(), dd.as<float>(), cn.as<uint32_t>(), sh.st);
        VDB_CUDA(cudaMemcpyAsync(r_ids.data(), ids.p, (size_t)nr * k * 8, cudaMemcpyDeviceToHost, sh.st));
        VDB_CUDA(cudaMemcpyAsync(r_dist.data(), dd.p, (size_t)nr * k * 4, cudaMemcpyDeviceToHost, sh.st));
        VDB_CUDA(cudaMemcpyAsync(r_cnt.data(), cn.p, (size_t)nr * 4, cudaMemcpyDeviceToHost, sh.st));
        VDB_CUDA(cudaStreamSynchronize(sh.st));
    });
    run_job(S, rp);
    int prev = 0;
    VDB_CUDA(cudaGetDevice(&prev));
    for (uint32_t i = 0; i < nr; ++i) {
        const uint32_t q = redo[i];
        if (host) {
            memcpy(a.h_ids + (size_t)q * k, r_ids.data() + (size_t)i * k, (size_t)k * 8);
            memcpy(a.h_dist + (size_t)q * k, r_dist.data() + (size_t)i * k, (size_t)k * 4);
            a.h_counts[q] = r_cnt[i];
        } else {
            const uint32_t h = q / per, r = q - h * per;
            VDB_CUDA(cudaSetDevice(S->shards[h].device));
            VDB_CUDA(cudaMemcpy(a.d_ids[h] + (size_t)r * k, r_ids.data() + (size_t)i * k, (size_t)k * 8, cudaMemcpyHostToDevice));
            VDB_CUDA(cudaMemcpy(a.d_dist[h] + (size_t)r * k, r_dist.data() + (size_t)i * k, (size_t)k * 4, cudaMemcpyHostToDevice));
            VDB_CUDA(cudaMemcpy(a.d_counts[h] + r, &r_cnt[i], 4, cudaMemcpyHostToDevice));
        }
    }
    VDB_CUDA(cudaSetDevice(prev));
}

static int effective_path(const vdb_dataset* md) { return md->flat_path >= 0 ? md->flat_path : g_flat_path.load(); }

// Queries per sharded Flat chunk. Above the fused top-k (the owners' merge runs in global memory) the per-shard keys and
// the owners' merge inputs, nq * k * 8 bytes each, stay within 1 GiB.
static uint32_t shard_query_chunk(uint32_t k) {
    if (merge_keys_fits(k)) return SHARD_QUERY_CHUNK;
    return (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(SHARD_QUERY_CHUNK, (1ull << 30) / ((uint64_t)k * 8)));
}

// IndexKNN::knn on the sharded set, host buffers (the call a Rust host makes, whatever the GPU count)
void sharded_flat_knn(const vdb_dataset* md, const void* queries, uint32_t nq, uint32_t k, uint64_t* ids, float* dist,
                      uint32_t* counts) {
    vdb_sharded_state* S = md->sharded;
    if (nq == 0) return;
    if (k == 0) {
        memset(counts, 0, (size_t)nq * 4);
        return;
    }
    std::lock_guard<std::mutex> lk(S->call_mu);
    const size_t rb = (size_t)md->dim * md->elem_size();
    const int path = effective_path(md);
    const uint32_t chunk = shard_query_chunk(k);
    for (uint32_t q0 = 0; q0 < nq; q0 += chunk) {
        FlatCallArgs a;
        a.nq = std::min(chunk, nq - q0);
        a.k = k;
        a.h_queries = (const uint8_t*)queries + (size_t)q0 * rb;
        a.h_ids = ids + (size_t)q0 * k;
        a.h_dist = dist + (size_t)q0 * k;
        a.h_counts = counts + q0;
        sharded_flat_chunk(md, a, path);
    }
}

// device-resident variant: d_queries[s] = the whole batch on shard s's device; shard s receives the results of the
// queries it owns, [lo_s, hi_s) with lo_s = s * ceil(nq / G), in d_ids[s] / d_dist[s] / d_counts[s]
void sharded_flat_knn_dev(const vdb_dataset* md, const void* const* d_queries, uint32_t nq, uint32_t k, uint64_t* const* d_ids,
                          float* const* d_dist, uint32_t* const* d_counts) {
    vdb_sharded_state* S = md->sharded;
    if (nq == 0) return;
    VDB_REQUIRE(k > 0, "k must be > 0");
    VDB_REQUIRE(nq <= SHARD_QUERY_CHUNK, "device-resident sharded search: at most %u queries per call", SHARD_QUERY_CHUNK);
    std::lock_guard<std::mutex> lk(S->call_mu);
    const uint32_t chunk = shard_query_chunk(k);
    if (nq <= chunk) {
        FlatCallArgs a;
        a.nq = nq;
        a.k = k;
        a.d_queries = d_queries;
        a.d_ids = d_ids;
        a.d_dist = d_dist;
        a.d_counts = d_counts;
        sharded_flat_chunk(md, a, effective_path(md));
        return;
    }
    // large k, more queries than one chunk: every chunk's owners write to their staging buffers, whose rows are then
    // copied to the owners of the whole call (query q -> shard q / per, row q % per)
    const uint32_t G = (uint32_t)S->shards.size(), per = ceil_div(nq, G);
    const size_t rb = (size_t)md->dim * md->elem_size();
    std::vector<const void*> qs(G);
    std::vector<uint64_t*> o_ids(G);
    std::vector<float*> o_dist(G);
    std::vector<uint32_t*> o_cnt(G);
    int prev = 0;
    VDB_CUDA(cudaGetDevice(&prev));
    for (uint32_t q0 = 0; q0 < nq; q0 += chunk) {
        const uint32_t cn = std::min(chunk, nq - q0), per_c = ceil_div(cn, G);
        for (uint32_t s = 0; s < G; ++s) {
            Shard& sh = S->shards[s];
            VDB_CUDA(cudaSetDevice(sh.device));
            sh.out_ids.ensure((size_t)per_c * k * 8);
            sh.out_dist.ensure((size_t)per_c * k * 4);
            sh.out_cnt.ensure((size_t)per_c * 4);
            qs[s] = (const uint8_t*)d_queries[s] + (size_t)q0 * rb;
            o_ids[s] = (uint64_t*)sh.out_ids.p;
            o_dist[s] = (float*)sh.out_dist.p;
            o_cnt[s] = (uint32_t*)sh.out_cnt.p;
        }
        VDB_CUDA(cudaSetDevice(prev));
        FlatCallArgs a;
        a.nq = cn;
        a.k = k;
        a.d_queries = qs.data();
        a.d_ids = o_ids.data();
        a.d_dist = o_dist.data();
        a.d_counts = o_cnt.data();
        sharded_flat_chunk(md, a, effective_path(md));   // ends with every shard's stream synchronised
        for (uint32_t hc = 0; hc < G; ++hc) {
            const uint32_t lo_c = std::min(cn, hc * per_c), hi_c = std::min(cn, (hc + 1) * per_c);
            for (uint32_t q = q0 + lo_c; q < q0 + hi_c;) {
                const uint32_t h = q / per, e = std::min(q0 + hi_c, (h + 1) * per), r = q - h * per, src = q - q0 - lo_c;
                const size_t n = e - q;
                VDB_CUDA(cudaMemcpy(d_ids[h] + (size_t)r * k, o_ids[hc] + (size_t)src * k, n * k * 8, cudaMemcpyDefault));
                VDB_CUDA(cudaMemcpy(d_dist[h] + (size_t)r * k, o_dist[hc] + (size_t)src * k, n * k * 4, cudaMemcpyDefault));
                VDB_CUDA(cudaMemcpy(d_counts[h] + r, o_cnt[hc] + src, n * 4, cudaMemcpyDefault));
                q = e;
            }
        }
    }
}

// ---- row-sharded IVF (SURVEY.md 8e): centroids replicated, every shard holds its slice of every list -------------------
vdb_ivf* sharded_ivf_create(const vdb_dataset* md, const void* h_centroids, uint32_t nlist, uint32_t* h_assign_out) {
    vdb_sharded_state* S = md->sharded;
    auto ivf = new vdb_ivf();
    ivf->device = md->device;
    ivf->nlist = nlist;
    ivf->dim = md->dim;
    ivf->dtype = md->dtype;
    ivf->metric = md->metric;
    ivf->n = md->n;
    ivf->parent = md;
    int prev = 0;
    cudaGetDevice(&prev);
    try {
        for (auto& sh : S->shards) {
            VDB_CUDA(cudaSetDevice(sh.device));
            ivf->shards.push_back(ivf_create(sh.ds, h_centroids, nlist, h_assign_out ? h_assign_out + sh.lo : nullptr));
        }
    } catch (...) {
        for (size_t i = 0; i < ivf->shards.size(); ++i) {
            cudaSetDevice(S->shards[i].device);
            ivf_destroy(ivf->shards[i]);
        }
        cudaSetDevice(prev);
        delete ivf;
        throw;
    }
    cudaSetDevice(prev);
    return ivf;
}

// the global lists: list l = the shards' slices of l in shard order (members ascending: shards are contiguous row blocks)
void sharded_ivf_lists(const vdb_dataset* md, const vdb_ivf* ivf, uint64_t* offsets, uint32_t* members) {
    vdb_sharded_state* S = md->sharded;
    const uint32_t G = (uint32_t)S->shards.size(), nlist = ivf->nlist;
    std::vector<std::vector<uint64_t>> off(G, std::vector<uint64_t>(nlist + 1));
    std::vector<std::vector<uint32_t>> mem(G);
    int prev = 0;
    VDB_CUDA(cudaGetDevice(&prev));
    for (uint32_t s = 0; s < G; ++s) {
        const vdb_ivf* sv = ivf->shards[s];
        VDB_CUDA(cudaSetDevice(S->shards[s].device));
        VDB_CUDA(cudaMemcpy(off[s].data(), sv->d_offsets, (size_t)(nlist + 1) * 8, cudaMemcpyDeviceToHost));
        mem[s].resize(sv->n);
        if (sv->n) VDB_CUDA(cudaMemcpy(mem[s].data(), sv->d_members, sv->n * 4, cudaMemcpyDeviceToHost));
    }
    VDB_CUDA(cudaSetDevice(prev));
    uint64_t at = 0;
    for (uint32_t l = 0; l < nlist; ++l) {
        offsets[l] = at;
        for (uint32_t s = 0; s < G; ++s)
            for (uint64_t i = off[s][l]; i < off[s][l + 1]; ++i) members[at++] = (uint32_t)(S->shards[s].lo + mem[s][i]);
    }
    offsets[nlist] = at;
}

// IndexKNNWithEf::knn_with_ef on the sharded set: every shard probes its slices of the n_probes nearest lists, the
// per-shard [nq, k] keys are merged by (distance, global id) on the queries' owners
void sharded_ivf_knn(const vdb_dataset* md, const vdb_ivf* ivf, const void* queries, uint32_t nq, uint32_t k, uint32_t n_probes,
                     uint64_t* ids, float* dist, uint32_t* counts) {
    vdb_sharded_state* S = md->sharded;
    if (nq == 0) return;
    if (k == 0) {
        memset(counts, 0, (size_t)nq * 4);
        return;
    }
    VDB_REQUIRE(ivf->shards.size() == S->shards.size(), "IVF index was not built on this sharded set");
    std::lock_guard<std::mutex> lk(S->call_mu);
    const size_t rb = (size_t)md->dim * md->elem_size();
    KeyProducer prod = [&](uint32_t s, const void* d_q, uint32_t n, uint32_t kk, uint64_t* d_keys, cudaStream_t st) {
        ivf_knn_keys(S->shards[s].ds, ivf->shards[s], d_q, n, kk, n_probes, d_keys, st);
    };
    for (uint32_t q0 = 0; q0 < nq; q0 += SHARD_QUERY_CHUNK) {
        FlatCallArgs a;
        a.nq = std::min(SHARD_QUERY_CHUNK, nq - q0);
        a.k = k;
        a.h_queries = (const uint8_t*)queries + (size_t)q0 * rb;
        a.h_ids = ids + (size_t)q0 * k;
        a.h_dist = dist + (size_t)q0 * k;
        a.h_counts = counts + q0;
        sharded_flat_chunk(md, a, 1, &prod);
    }
}

// ---- row-sharded PQ (SURVEY.md 8e) -------------------------------------------------------------------------------------
vdb_pq* sharded_pq_create(const vdb_dataset* md, const void* h_codebooks, uint32_t m, uint32_t n_bits, const uint8_t* h_codes_in,
                          uint8_t* h_codes_out) {
    vdb_sharded_state* S = md->sharded;
    auto pq = new vdb_pq();
    pq->device = md->device;
    pq->dim = md->dim;
    pq->dtype = md->dtype;
    pq->metric = md->metric;
    pq->n = md->n;
    pq->m = m;
    pq->n_bits = n_bits;
    int prev = 0;
    cudaGetDevice(&prev);
    try {
        for (auto& sh : S->shards) {
            VDB_CUDA(cudaSetDevice(sh.device));
            const size_t enc = n_bits == 4 ? (m + 1) / 2 : m;
            pq->shards.push_back(pq_create(sh.ds, h_codebooks, m, n_bits, h_codes_in ? h_codes_in + sh.lo * enc : nullptr,
                                           h_codes_out ? h_codes_out + sh.lo * enc : nullptr));
            pq->enc = pq->shards.back()->enc;
            pq->kc = pq->shards.back()->kc;
        }
    } catch (...) {
        for (size_t i = 0; i < pq->shards.size(); ++i) {
            cudaSetDevice(S->shards[i].device);
            pq_destroy(pq->shards[i]);
        }
        cudaSetDevice(prev);
        delete pq;
        throw;
    }
    cudaSetDevice(prev);
    pq->serial = pq->shards.front()->serial;   // unique: shard tables are never handed out on their own
    pq->parent = md;
    return pq;
}

// IndexPQ::knn_pq on the sharded set (Flat, or IVF restricted to the probed lists), identical to the unsharded call:
// (1) every shard's max(ef, k) best codes by (ADC, global id) - `candidates` - go to the queries' owners, (2) the owners
// merge them into the GLOBAL top-max(ef, k) and peer-store their slice of it into every shard, (3) every shard reranks
// exactly the candidates it owns, (4) the [nq, k] keys are merged on the owners.
static void sharded_knn_pq(const vdb_dataset* md, const void* queries, uint32_t nq, uint32_t k, uint32_t ef, uint64_t* ids,
                           float* dist, uint32_t* counts, const KeyProducer& candidates) {
    vdb_sharded_state* S = md->sharded;
    if (nq == 0) return;
    if (k == 0) {
        memset(counts, 0, (size_t)nq * 4);
        return;
    }
    VDB_REQUIRE(nq <= SHARD_QUERY_CHUNK, "sharded knn_pq: at most %u queries per call", SHARD_QUERY_CHUNK);
    std::lock_guard<std::mutex> lk(S->call_mu);
    const uint32_t G = (uint32_t)S->shards.size(), kk = std::max(ef, k);
    const size_t rb = (size_t)md->dim * md->elem_size();
    const uint32_t per = ceil_div(nq, G);
    auto slice = [&](uint32_t h, uint32_t* lo, uint32_t* hi) {
        *lo = std::min(nq, h * per);
        *hi = std::min(nq, (h + 1) * per);
    };
    {
        int prev = 0;
        VDB_CUDA(cudaGetDevice(&prev));
        for (uint32_t s = 0; s < G; ++s) {
            Shard& sh = S->shards[s];
            uint32_t lo, hi;
            slice(s, &lo, &hi);
            const uint32_t cnt = std::max(hi - lo, 1u);
            VDB_CUDA(cudaSetDevice(sh.device));
            sh.q_all.ensure((size_t)nq * rb);
            sh.kin.ensure((size_t)G * cnt * kk * 8);
            sh.jall.ensure((size_t)nq * kk * 8);          // the global candidate lists, written by the owners
            sh.out_ids.ensure((size_t)cnt * k * 8);
            sh.out_dist.ensure((size_t)cnt * k * 4);
            sh.out_cnt.ensure((size_t)cnt * 4);
        }
        VDB_CUDA(cudaSetDevice(prev));
    }
    std::vector<DevBuf> keys(G), merged(G);
    std::vector<std::function<void(uint32_t)>> ph;
    ph.push_back([&](uint32_t s) {   // queries: every shard uploads the batch (knn_pq batches are small next to the code scan)
        Shard& sh = S->shards[s];
        VDB_CUDA(cudaMemcpyAsync(sh.q_all.p, queries, (size_t)nq * rb, cudaMemcpyHostToDevice, sh.st));
        keys[s] = DevBuf((size_t)nq * kk * 8, sh.st);
        candidates(s, sh.q_all.p, nq, kk, keys[s].as<uint64_t>(), sh.st);
        PtrList dk{}, df{};
        for (uint32_t h = 0; h < G; ++h) {
            uint32_t lo, hi;
            slice(h, &lo, &hi);
            dk.p[h] = (uint8_t*)S->shards[h].kin.p + (size_t)s * std::max(hi - lo, 1u) * kk * 8;
        }
        scatter_owner_kernel<<<nq, 128, 0, sh.st>>>(keys[s].as<uint64_t>(), nullptr, nq, kk, per, dk, df);
        VDB_LAUNCHED();
        VDB_CUDA(cudaEventRecord(sh.ev[EV_S], sh.st));
    });
    ph.push_back([&](uint32_t s) {   // owners: global top-kk of their queries, peer-stored into every shard
        Shard& sh = S->shards[s];
        wait_peers(S, s, EV_S);
        uint32_t lo, hi;
        slice(s, &lo, &hi);
        const uint32_t cnt = hi - lo;
        if (cnt) {
            merged[s] = DevBuf((size_t)cnt * kk * 8, sh.st);
            launch_merge_sorted((const uint64_t*)sh.kin.p, G, cnt, kk, kk, merged[s].as<uint64_t>(), nullptr, nullptr, nullptr, sh.st);
            PtrList dst{};
            for (uint32_t h = 0; h < G; ++h) dst.p[h] = (uint8_t*)S->shards[h].jall.p + (size_t)lo * kk * 8;
            bcast(merged[s].p, (size_t)cnt * kk * 8, dst, G, sh.st);
        }
        VDB_CUDA(cudaEventRecord(sh.ev[EV_Q], sh.st));
    });
    ph.push_back([&](uint32_t s) {   // exact rerank of the candidates this shard owns
        Shard& sh = S->shards[s];
        wait_peers(S, s, EV_Q);
        keys[s] = DevBuf((size_t)nq * k * 8, sh.st);
        rerank_keys(sh.ds, sh.q_all.p, nq, (const uint64_t*)sh.jall.p, kk, k, keys[s].as<uint64_t>(), sh.st);
        PtrList dk{}, df{};
        for (uint32_t h = 0; h < G; ++h) {
            uint32_t lo, hi;
            slice(h, &lo, &hi);
            dk.p[h] = (uint8_t*)S->shards[h].kin.p + (size_t)s * std::max(hi - lo, 1u) * k * 8;
        }
        // kin is reused for the second exchange: every shard has finished reading its first contents (it waited for
        // EV_Q of all peers, which they record after their merge of phase 2)
        scatter_owner_kernel<<<nq, 128, 0, sh.st>>>(keys[s].as<uint64_t>(), nullptr, nq, k, per, dk, df);
        VDB_LAUNCHED();
        VDB_CUDA(cudaEventRecord(sh.ev[EV_F], sh.st));
    });
    ph.push_back([&](uint32_t s) {
        Shard& sh = S->shards[s];
        wait_peers(S, s, EV_F);
        uint32_t lo, hi;
        slice(s, &lo, &hi);
        const uint32_t cnt = hi - lo;
        if (cnt) {
            launch_merge_sorted((const uint64_t*)sh.kin.p, G, cnt, k, k, nullptr, (uint64_t*)sh.out_ids.p, (float*)sh.out_dist.p,
                                (uint32_t*)sh.out_cnt.p, sh.st);
            VDB_CUDA(cudaMemcpyAsync(ids + (size_t)lo * k, sh.out_ids.p, (size_t)cnt * k * 8, cudaMemcpyDeviceToHost, sh.st));
            VDB_CUDA(cudaMemcpyAsync(dist + (size_t)lo * k, sh.out_dist.p, (size_t)cnt * k * 4, cudaMemcpyDeviceToHost, sh.st));
            VDB_CUDA(cudaMemcpyAsync(counts + lo, sh.out_cnt.p, (size_t)cnt * 4, cudaMemcpyDeviceToHost, sh.st));
        }
        keys[s] = DevBuf();
        merged[s] = DevBuf();
        VDB_CUDA(cudaStreamSynchronize(sh.st));
    });
    run_job(S, ph);
}

void sharded_pq_knn(const vdb_dataset* md, const vdb_pq* pq, const void* queries, uint32_t nq, uint32_t k, uint32_t ef,
                    uint64_t* ids, float* dist, uint32_t* counts) {
    vdb_sharded_state* S = md->sharded;
    VDB_REQUIRE(nq == 0 || k == 0 || pq->shards.size() == S->shards.size(), "PQ table was not built on this sharded set");
    sharded_knn_pq(md, queries, nq, k, ef, ids, dist, counts,
                   [&](uint32_t s, const void* d_q, uint32_t n, uint32_t kk, uint64_t* d_keys, cudaStream_t st) {
                       pq_adc_keys(S->shards[s].ds, pq->shards[s], d_q, n, kk, d_keys, st);
                   });
}

void sharded_ivf_knn_pq(const vdb_dataset* md, const vdb_ivf* ivf, const vdb_pq* pq, const void* queries, uint32_t nq, uint32_t k,
                        uint32_t ef, uint32_t n_probes, uint64_t* ids, float* dist, uint32_t* counts) {
    vdb_sharded_state* S = md->sharded;
    VDB_REQUIRE(ivf->shards.size() == S->shards.size() && ivf->parent == md && ivf->n == md->n,
                "IVF index was built for a different vector set");
    VDB_REQUIRE(pq->shards.size() == S->shards.size() && pq->n == md->n,
                "PQ table was built for a different vector set (it must be rebuilt after add/delete)");
    VDB_REQUIRE(n_probes > 0, "The number of probes should be greater than 0.");
    sharded_knn_pq(md, queries, nq, k, ef, ids, dist, counts,
                   [&](uint32_t s, const void* d_q, uint32_t n, uint32_t kk, uint64_t* d_keys, cudaStream_t st) {
                       ivf_pq_adc_keys(S->shards[s].ds, ivf->shards[s], pq->shards[s], d_q, n, kk, n_probes, d_keys, st);
                   });
}

// ---- HNSW on a row-sharded set (DESIGN.md section 6): one full replica per shard entry ---------------------------------
// A graph walk reads whichever rows the previous hop leads to, so HNSW is replicated, not sharded: replica r holds all n
// rows and the same graph on shard r's device. A search splits its batch into contiguous slices, one per replica, and each
// slice runs the single-GPU search on its replica: results are bit-identical to the unsharded index.
vdb_dataset* adopt_dataset_on(int device, const void* d_rows, uint64_t n, uint32_t dim, uint32_t pitch, int dtype, int metric,
                              uint64_t id_base);   // capi.cu
cudaStream_t thread_stream();                      // capi.cu: the calling thread's stream on the current device

}  // namespace vdb

struct HnswPqReplicas {
    uint64_t serial = 0;         // vdb_pq::serial of the row-sharded table the codes come from
    std::vector<vdb_pq*> pq;     // pq[r]: the table's codebooks and the codes of all n rows on replica r's device
    ~HnswPqReplicas() {
        int prev = 0;
        cudaGetDevice(&prev);
        for (vdb_pq* t : pq) {
            cudaSetDevice(t->device);
            vdb::pq_destroy(t);
        }
        cudaSetDevice(prev);
    }
};

namespace vdb {

namespace {
struct KeepDevice {   // restores the calling thread's current device on every way out
    int prev = 0;
    KeepDevice() { VDB_CUDA(cudaGetDevice(&prev)); }
    ~KeepDevice() { cudaSetDevice(prev); }
};
}  // namespace

static void free_replicas(HnswReplicas* rep) {
    KeepDevice kd;
    rep->pq.reset();
    for (size_t r = 0; r < rep->ds.size(); ++r) {
        cudaSetDevice(rep->ds[r]->device);
        if (r < rep->h.size()) hnsw_destroy(rep->h[r]);
        vdb_dataset_destroy(rep->ds[r]);
    }
    delete rep;
}

// the replicas' rows: every shard's row block is peer-copied into one buffer of all n rows on each shard entry's device
static HnswReplicas* replicate_rows(const vdb_dataset* md) {
    vdb_sharded_state* S = md->sharded;
    const uint32_t G = (uint32_t)S->shards.size();
    const uint32_t pitch = S->shards[0].ds->pitch;   // one pitch for every shard (vdb_dataset_create / _create_sharded_dev)
    const size_t pb = (size_t)pitch * md->elem_size();
    KeepDevice kd;
    auto rep = new HnswReplicas();
    rep->parent = md;
    std::vector<cudaStream_t> st;
    try {
        for (uint32_t r = 0; r < G; ++r) {
            const int dev = S->shards[r].device;
            VDB_CUDA(cudaSetDevice(dev));
            void* buf = nullptr;
            VDB_CUDA(cudaMalloc(&buf, std::max<uint64_t>(md->n, 1) * pb));
            vdb_dataset* ds = nullptr;
            try {
                ds = adopt_dataset_on(dev, buf, md->n, md->dim, pitch, md->dtype, md->metric, md->id_base);
            } catch (...) {
                cudaFree(buf);
                throw;
            }
            ds->owned = true;   // vdb_dataset_destroy frees the buffer
            rep->ds.push_back(ds);
            st.push_back(thread_stream());
            for (const Shard& sh : S->shards)
                if (sh.hi > sh.lo)
                    VDB_CUDA(cudaMemcpyPeerAsync((uint8_t*)buf + sh.lo * pb, dev, sh.ds->d_rows, sh.device, (sh.hi - sh.lo) * pb, st[r]));
        }
        for (uint32_t r = 0; r < G; ++r) {
            VDB_CUDA(cudaSetDevice(rep->ds[r]->device));
            VDB_CUDA(cudaStreamSynchronize(st[r]));
        }
    } catch (...) {
        for (size_t r = 0; r < st.size(); ++r) {
            cudaSetDevice(rep->ds[r]->device);
            cudaStreamSynchronize(st[r]);
        }
        free_replicas(rep);
        throw;
    }
    return rep;
}

// replicas rep->h.size() .. G-1 from a graph in host memory (the layouts of vdb_hnsw_create_from_graph)
static void replicate_graph(HnswReplicas* rep, uint32_t M, uint32_t ef_construction, const uint32_t* h_levels, const uint32_t* links0,
                            const uint32_t* len0, const uint32_t* ulinks, const uint32_t* ulen, int64_t enter_point,
                            int32_t enter_level) {
    for (size_t r = rep->h.size(); r < rep->ds.size(); ++r) {
        VDB_CUDA(cudaSetDevice(rep->ds[r]->device));
        rep->h.push_back(hnsw_from_graph(rep->ds[r], M, ef_construction, h_levels, links0, len0, ulinks, ulen, enter_point,
                                         enter_level));
    }
}

// the caller's handle: replica 0's scalars, no arrays of its own
static vdb_hnsw* replicated_handle(HnswReplicas* rep) {
    const vdb_hnsw* h0 = rep->h[0];
    auto h = new vdb_hnsw();
    h->device = h0->device;
    h->n = h0->n;
    h->dim = h0->dim;
    h->dtype = h0->dtype;
    h->metric = h0->metric;
    h->M = h0->M;
    h->M0 = h0->M0;
    h->ef_construction = h0->ef_construction;
    h->h_level = h0->h_level;
    h->slots = h0->slots;
    h->enter_point = h0->enter_point;
    h->enter_level = h0->enter_level;
    h->rep = rep;
    return h;
}

// build once on replica 0, then every other replica loads that graph
vdb_hnsw* sharded_hnsw_build(const vdb_dataset* md, uint32_t M, uint32_t ef_construction, const uint32_t* h_levels,
                             uint32_t max_batch) {
    KeepDevice kd;
    HnswReplicas* rep = replicate_rows(md);
    try {
        VDB_CUDA(cudaSetDevice(rep->ds[0]->device));
        rep->h.push_back(hnsw_build(rep->ds[0], M, ef_construction, h_levels, max_batch));
        const vdb_hnsw* h0 = rep->h[0];
        const uint64_t n = h0->n;
        std::vector<uint32_t> links0(n * h0->M0), len0(n), ulinks(h0->slots * h0->M), ulen(h0->slots);
        if (n) {
            VDB_CUDA(cudaMemcpy(links0.data(), h0->d_links0, links0.size() * 4, cudaMemcpyDeviceToHost));
            VDB_CUDA(cudaMemcpy(len0.data(), h0->d_len0, len0.size() * 4, cudaMemcpyDeviceToHost));
        }
        if (h0->slots) {
            VDB_CUDA(cudaMemcpy(ulinks.data(), h0->d_ulinks, ulinks.size() * 4, cudaMemcpyDeviceToHost));
            VDB_CUDA(cudaMemcpy(ulen.data(), h0->d_ulen, ulen.size() * 4, cudaMemcpyDeviceToHost));
        }
        replicate_graph(rep, h0->M, h0->ef_construction, h0->h_level.data(), links0.data(), len0.data(), ulinks.data(), ulen.data(),
                        h0->enter_point, h0->enter_level);
    } catch (...) {
        free_replicas(rep);
        throw;
    }
    return replicated_handle(rep);
}

vdb_hnsw* sharded_hnsw_from_graph(const vdb_dataset* md, uint32_t M, uint32_t ef_construction, const uint32_t* h_levels,
                                  const uint32_t* links0, const uint32_t* len0, const uint32_t* ulinks, const uint32_t* ulen,
                                  int64_t enter_point, int32_t enter_level) {
    KeepDevice kd;
    HnswReplicas* rep = replicate_rows(md);
    try {
        replicate_graph(rep, M, ef_construction, h_levels, links0, len0, ulinks, ulen, enter_point, enter_level);
    } catch (...) {
        free_replicas(rep);
        throw;
    }
    return replicated_handle(rep);
}

void sharded_hnsw_destroy(vdb_hnsw* h) {
    free_replicas(h->rep);
    delete h;
}

// one unsharded table per replica from a row-sharded table: the same codebooks, the shards' codes in row order
static std::shared_ptr<const HnswPqReplicas> pq_replicas(HnswReplicas* rep, const vdb_pq* pq) {
    std::lock_guard<std::mutex> lk(rep->pq_mu);
    if (rep->pq && rep->pq->serial == pq->serial) return rep->pq;
    const vdb_pq* t0 = pq->shards[0];
    std::vector<uint8_t> books((size_t)t0->kc * t0->dim * (t0->dtype == VDB_F32 ? 4 : 1));   // groups partition the dims
    std::vector<uint8_t> codes(std::max<uint64_t>(pq->n * pq->enc, 1));
    VDB_CUDA(cudaSetDevice(t0->device));
    VDB_CUDA(cudaMemcpy(books.data(), t0->d_codebooks, books.size(), cudaMemcpyDeviceToHost));
    uint64_t at = 0;
    for (const vdb_pq* t : pq->shards) {
        VDB_CUDA(cudaSetDevice(t->device));
        if (t->n) VDB_CUDA(cudaMemcpy(codes.data() + at * pq->enc, t->d_codes, t->n * t->enc, cudaMemcpyDeviceToHost));
        at += t->n;
    }
    auto c = std::make_shared<HnswPqReplicas>();
    c->serial = pq->serial;
    for (vdb_dataset* ds : rep->ds) {
        VDB_CUDA(cudaSetDevice(ds->device));
        c->pq.push_back(pq_create(ds, books.data(), pq->m, pq->n_bits, codes.data(), nullptr));
    }
    rep->pq = c;
    return c;
}

// knn_with_ef (pq == nullptr) / knn_pq on the sharded set: min(G, nq) contiguous slices of the batch, slice i on replica
// (first + i) % G. Every slice's upload, search and download is enqueued on the calling thread's stream of its replica's
// device before any is waited for, so the replicas run at the same time; the call stays re-entrant (no shared state
// but the replicas' overflow / evaluation counters, which are atomics).
void sharded_hnsw_knn(const vdb_dataset* md, const vdb_hnsw* h, const vdb_pq* pq, const void* queries, uint32_t nq, uint32_t k,
                      uint32_t ef, uint64_t* ids, float* dist, uint32_t* counts) {
    HnswReplicas* rep = h->rep;
    VDB_REQUIRE(rep && rep->parent == md && h->n == md->n, "HNSW index was built for a different vector set");
    if (pq) {
        VDB_REQUIRE(!pq->shards.empty() && pq->parent == md && pq->n == md->n,
                    "PQ table was built for a different vector set (it must be rebuilt after add/delete)");
        VDB_REQUIRE(pq->metric == md->metric, "Distance algorithm mismatch.");
        VDB_REQUIRE(pq->n_bits == 4, "HNSW + PQ search supports 4-bit codes");
    }
    if (nq == 0) return;
    if (k == 0) {
        memset(counts, 0, (size_t)nq * 4);
        return;
    }
    KeepDevice kd;
    const std::shared_ptr<const HnswPqReplicas> pqr = pq ? pq_replicas(rep, pq) : nullptr;
    const uint32_t G = (uint32_t)rep->h.size(), R = std::min(G, nq);
    // calls with fewer queries than replicas start at a rotating replica, so concurrent single-query callers spread out
    const uint32_t first = nq < G ? rep->next.fetch_add(1, std::memory_order_relaxed) % G : 0;
    const size_t rb = (size_t)md->dim * md->elem_size();
    struct Slice {
        uint32_t r = 0, lo = 0, cnt = 0;
        cudaStream_t st = nullptr;
        DevBuf q, keys, ids, dist, counts;
    };
    std::vector<Slice> sl(R);
    auto settle = [&](Slice& x) {   // waits for the slice and frees its buffers on its device
        VDB_CUDA(cudaSetDevice(rep->ds[x.r]->device));
        VDB_CUDA(cudaStreamSynchronize(x.st));
        x.q = DevBuf();
        x.keys = DevBuf();
        x.ids = DevBuf();
        x.dist = DevBuf();
        x.counts = DevBuf();
    };
    try {
        for (uint32_t i = 0; i < R; ++i) {
            Slice& x = sl[i];
            uint64_t lo, hi;
            shard_bounds(nq, R, i, &lo, &hi);
            x.r = (first + i) % G;
            x.lo = (uint32_t)lo;
            x.cnt = (uint32_t)(hi - lo);
            const vdb_dataset* ds = rep->ds[x.r];
            VDB_CUDA(cudaSetDevice(ds->device));
            x.st = thread_stream();
            x.q = DevBuf((size_t)x.cnt * rb, x.st);
            x.keys = DevBuf((size_t)x.cnt * k * 8, x.st);
            x.ids = DevBuf((size_t)x.cnt * k * 8, x.st);
            x.dist = DevBuf((size_t)x.cnt * k * 4, x.st);
            x.counts = DevBuf((size_t)x.cnt * 4, x.st);
            VDB_CUDA(cudaMemcpyAsync(x.q.p, (const uint8_t*)queries + (size_t)x.lo * rb, (size_t)x.cnt * rb, cudaMemcpyHostToDevice,
                                     x.st));
            if (pq) hnsw_knn_pq_keys(ds, rep->h[x.r], pqr->pq[x.r], x.q.p, x.cnt, k, ef, x.keys.as<uint64_t>(), x.st);
            else hnsw_knn_keys(ds, rep->h[x.r], x.q.p, x.cnt, k, ef, x.keys.as<uint64_t>(), x.st);
            decode_keys(x.keys.as<uint64_t>(), x.cnt, k, x.ids.as<uint64_t>(), x.dist.as<float>(), x.counts.as<uint32_t>(), x.st);
        }
        for (Slice& x : sl) {
            VDB_CUDA(cudaSetDevice(rep->ds[x.r]->device));
            VDB_CUDA(cudaMemcpyAsync(ids + (size_t)x.lo * k, x.ids.p, (size_t)x.cnt * k * 8, cudaMemcpyDeviceToHost, x.st));
            VDB_CUDA(cudaMemcpyAsync(dist + (size_t)x.lo * k, x.dist.p, (size_t)x.cnt * k * 4, cudaMemcpyDeviceToHost, x.st));
            VDB_CUDA(cudaMemcpyAsync(counts + x.lo, x.counts.p, (size_t)x.cnt * 4, cudaMemcpyDeviceToHost, x.st));
        }
    } catch (...) {
        for (Slice& x : sl)   // nothing enqueued by the call may outlive it
            if (x.st) {
                cudaSetDevice(rep->ds[x.r]->device);
                cudaStreamSynchronize(x.st);
            }
        throw;
    }
    // every replica that took part has its counter read (and cleared); a full visited set on any of them fails the call
    int code = 0;
    std::string err;
    for (Slice& x : sl) {
        settle(x);
        try {
            hnsw_check_overflow(rep->h[x.r], x.st);
        } catch (const Error& e) {
            if (!code) code = e.code, err = e.what();
        }
    }
    if (code) throw Error(code, err);
}

uint32_t sharded_count(const vdb_dataset* md) { return md->sharded ? (uint32_t)md->sharded->shards.size() : 0; }
void sharded_info(const vdb_dataset* md, uint32_t s, int* device, uint64_t* lo, uint64_t* hi, vdb_dataset** ds) {
    VDB_REQUIRE(md->sharded && s < md->sharded->shards.size(), "shard %u out of range", s);
    const Shard& sh = md->sharded->shards[s];
    if (device) *device = sh.device;
    if (lo) *lo = sh.lo;
    if (hi) *hi = sh.hi;
    if (ds) *ds = sh.ds;
}

}  // namespace vdb
