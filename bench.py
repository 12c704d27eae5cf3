#!/usr/bin/env python
"""bench.py — headline benchmark of the search hot path (BASELINE.json: QPS, 1Mx960 Flat L2 kNN).

    python bench.py [--gpus N] [--steps K] [--warmup W]            our arm (CUDA kernels)
    python bench.py [...] --dump-outputs DIR                        also write the last timed step's results as .npy
    python bench.py --impl reference [...]                          CPU arm: the oracle (reference
                                                                    semantics restated in C++; the Rust
                                                                    crate cannot be built in this image)

Workload (configs[1] of BASELINE.json): synthetic GIST-shaped 1,000,000 x 960 f32 database,
10,000-query batch, k = 100, L2Sqr, exact Flat search; rows are sharded over the N GPUs (strong
scaling) and per-GPU top-k lists are merged after one NCCL all-gather. One "step" = one pass of the
whole query batch. Prints ONE JSON line (rank 0).
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DIM = 960
GEMM_PASS_TRAFFIC = 1.952671e9 + 45.116e6  # dram__bytes_read.sum + dram__bytes_write.sum of ONE filter launch (the whole pass:
#                                            1M x 960 FP16 operand rows, 10 000 queries): end-of-round re-capture of the
#                                            shipped kernel, profiles/r02_flat_gemm_ncu.md (first capture: 1.954014e9 + 45.709e6)
CHUNK = 50_000  # rows per generator chunk (seeded per chunk so any sharding sees the same bits)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--nq", type=int, default=10_000)
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--path", default="auto", choices=["auto", "scan", "tensor"])
    ap.add_argument("--cpu-queries", type=int, default=0, help="CPU sample size (0 = 2 x cores, <= 128)")
    ap.add_argument("--no-other-configs", action="store_true",
                    help="skip the IVF (configs[2]) and PQ (configs[3]) legs that follow the headline measurement at N=1")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_BYTES = 64 << 20  # --dump-outputs: bound on all written arrays together


def dump_outputs(out_dir, ids, dist, counts):
    """The search results of the last timed step, as the caller of the timed path receives them, as DIR/<name>.npy:
    ids and counts in float64 (exact below 2^53; an unfilled id slot reads -1), distances in float32. When the whole
    batch is larger than DUMP_BYTES, a fixed seeded sample of the queries is written; query_rows.npy always names the
    query rows written, so that two builds can be compared output for output."""
    ids = np.asarray(ids).astype(np.int64).astype(np.float64)
    dist = np.asarray(dist, np.float32)
    counts = np.asarray(counts).astype(np.float64)
    nq, k = ids.shape
    rows = np.arange(nq)
    per_query = k * (8 + 4) + 8 + 8
    if nq * per_query > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(nq, DUMP_BYTES // per_query, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("ids", ids[rows]), ("dist", dist[rows]), ("counts", counts[rows]),
                    ("query_rows", rows.astype(np.float64))):
        np.save(os.path.join(out_dir, name + ".npy"), a)


def load_fixtures():
    fx = np.load(os.path.join(ROOT, "tests", "golden", "fixtures.npz"))
    dec = lambda u: (u.astype(np.float64) / 1e4).astype(np.float32)  # noqa: E731
    return dec(fx["base_u16"]), dec(fx["test_u16"])


def synth(proto, lo, hi, seed, dev):
    """Rows [lo, hi) of the synthetic set: proto[i % 1000] + 0.02 * N(0,1), clamped to [0,1] and rounded to
    the 1e-4 grid of the real GIST data (SURVEY.md section 8d). Generated on the GPU, chunk-seeded."""
    import torch
    out = torch.empty((hi - lo, DIM), dtype=torch.float32, device=dev)
    proto = torch.as_tensor(proto, device=dev)
    c = lo // CHUNK
    while c * CHUNK < hi:
        c_lo, c_hi = c * CHUNK, (c + 1) * CHUNK
        g = torch.Generator(device=dev)
        g.manual_seed(seed * 1_000_003 + c)
        z = torch.randn((CHUNK, DIM), generator=g, device=dev, dtype=torch.float32)
        a, b = max(lo, c_lo), min(hi, c_hi)
        idx = torch.arange(a, b, device=dev) % proto.shape[0]
        x = proto[idx] + 0.02 * z[a - c_lo:b - c_lo]
        out[a - lo:b - lo] = torch.round(x.clamp_(0.0, 1.0) * 1e4) / 1e4
        del z
        c += 1
    return out


def synth_clustered(proto, lo, hi, seed, dev, latent=32, spread=0.010, noise=0.018):
    """Second synthetic set for the recall-calibrated legs (IVF / PQ / HNSW): rows [lo, hi) of a mixture of LOW-RANK
    clouds. Row i = prototype i % 1000 + L z_i + isotropic noise, z_i ~ N(0, 1)^latent, L a fixed [latent, 960] matrix
    giving a per-dimension standard deviation `spread`; clamped to [0, 1] on the 1e-4 grid of the real GIST data. Inside
    a prototype's cloud the distances now vary with the latent coordinates (relative contrast ~2 between the nearest
    neighbours and a typical member, as in real descriptors), whereas the flat set of bench.synth has 1000
    near-equidistant copies per prototype that PQ / HNSW can only rank by chance (recall ~ ef / 1000)."""
    import torch
    proto = torch.as_tensor(proto, device=dev)
    g = torch.Generator(device=dev)
    g.manual_seed(977)                      # L depends on nothing but this constant
    lmat = torch.randn((latent, DIM), generator=g, device=dev) * (spread / latent ** 0.5)
    out = torch.empty((hi - lo, DIM), dtype=torch.float32, device=dev)
    c = lo // CHUNK
    while c * CHUNK < hi:
        c_lo, c_hi = c * CHUNK, (c + 1) * CHUNK
        g2 = torch.Generator(device=dev)
        g2.manual_seed(seed * 1_000_003 + c)
        z = torch.randn((CHUNK, DIM), generator=g2, device=dev, dtype=torch.float32)
        zl = torch.randn((CHUNK, latent), generator=g2, device=dev, dtype=torch.float32)
        a, b = max(lo, c_lo), min(hi, c_hi)
        idx = torch.arange(a, b, device=dev) % proto.shape[0]
        x = proto[idx] + zl[a - c_lo:b - c_lo] @ lmat + noise * z[a - c_lo:b - c_lo]
        out[a - lo:b - lo] = torch.round(x.clamp_(0.0, 1.0) * 1e4) / 1e4
        del z, zl
        c += 1
    return out


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "50", "-i", str(index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def wait_ready(self, timeout=5.0):
        """Blocks until the first sample is out: nvidia-smi's start-up (NVML initialisation, ~0.3 s) can stall the CUDA
        driver calls of this process for tens of milliseconds and must not overlap the timed steps (seen once as a 85 ms
        gap in a 1-step run)."""
        if self.p is None:
            return
        t0 = time.perf_counter()
        while time.perf_counter() - t0 < timeout and self.p.poll() is None:
            try:
                if os.path.getsize(self.f.name) > 0:
                    return
            except OSError:
                return
            time.sleep(0.02)

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [s.strip() for s in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.f.name)
        if sm:
            # under-load samples only: drop the idle head/tail
            hot = [s for s in sm if s >= 0.5 * max(sm)]
            out = {"sm_mhz": statistics.median(hot), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                   "samples": len(sm)}
        return out


def cpu_arm(base_host, q_host, k, cores, steps, warmup, gpu_check=None):
    """Times the oracle (reference semantics) on `q_host` with all host threads. Returns (qps, results)."""
    import oracle as O
    O.lib()
    res = None
    for _ in range(warmup):
        res = O.flat_knn(base_host, q_host[:max(1, min(len(q_host), cores))], k, "l2sqr", cores)
    t0 = time.perf_counter()
    for _ in range(steps):
        res = O.flat_knn(base_host, q_host, k, "l2sqr", cores)
    dt = (time.perf_counter() - t0) / steps
    return len(q_host) / dt, dt, res


def measure_tf32_peak(dev, seconds=1.5):
    """cuBLAS TF32 GEMM 8192^3 on this GPU: burst (best of 10) and sustained (back to back). MEASURED_PEAKS.json
    has no TF32 figure, so the roofline denominator for the TF32 contraction is measured here, next to the kernel."""
    import torch
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        n = 8192
        a = torch.randn((n, n), device=dev)
        b = torch.randn((n, n), device=dev)
        for _ in range(3):
            a @ b
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            a @ b
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        burst = 2.0 * n ** 3 / (best * 1e-3) / 1e12
        reps = 0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        while time.perf_counter() - t0 < seconds:
            for _ in range(20):
                a @ b
            reps += 20
            torch.cuda.synchronize()
        e1.record()
        torch.cuda.synchronize()
        sustained = 2.0 * n ** 3 * reps / (e0.elapsed_time(e1) * 1e-3) / 1e12
        return burst, sustained
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


def tensor_peak(dev, peaks, f16):
    """Roofline denominator of the contraction. FP16 operands: the driver-written dense bf16 figure of
    MEASURED_PEAKS.json (fp16 and bf16 share the tensor rate), sustained - the kernel is timed inside a long step.
    TF32 operands: MEASURED_PEAKS.json has no TF32 figure, so cuBLAS TF32 8192^3 is measured here, next to the kernel."""
    if f16 and peaks.get("bf16_tflops_sustained"):
        return (peaks["bf16_tflops_sustained"],
                "MEASURED_PEAKS.json bf16_tflops_sustained (driver-written; burst %.1f)" % (peaks.get("bf16_tflops") or 0.0))
    if f16:
        return 1403.0, "fallback: B200_PROFILING.md sustained dense bf16 figure (MEASURED_PEAKS.json absent)"
    burst, sustained = measure_tf32_peak(dev)
    return sustained, ("cuBLAS TF32 8192^3 measured in this run, sustained (burst %.1f); nominal dense TF32 is 1100; "
                       "MEASURED_PEAKS.json has bf16 only (%.1f sustained)" % (burst, peaks.get("bf16_tflops_sustained") or 0.0))


def tensor_stats(lib, ds_handle=None):
    q, c, f = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
    lib.vdb_flat_gemm_stats(C.byref(q), C.byref(c), C.byref(f))
    if q.value == 0:
        return None
    out = {"queries": q.value, "candidates_per_query": c.value / q.value, "exact_fallback_queries": f.value}
    if ds_handle is not None:
        kind, scale, mn, me, sb = C.c_int(-1), C.c_float(0), C.c_float(0), C.c_float(0), C.c_uint64(0)
        if lib.vdb_dataset_operand_info(ds_handle, C.byref(kind), C.byref(scale), C.byref(mn), C.byref(me), C.byref(sb)) == 0:
            out["operand"] = {"kind": {0: "tf32 (fp32 rows in place, hardware truncation)", 1: "fp16 copy (power-of-two scaled)"}.get(kind.value, "not built"),
                              "scale": scale.value, "mean_row_norm": mn.value, "mean_operand_error_norm": me.value,
                              "side_array_bytes": sb.value}
    return out


def single_query_e2e(flat, q_host, n_rows, peak_gbs, k=10):
    """vdb_flat_knn with nq = 1 and HOST pointers from T native caller threads on one handle (the reference searches
    one query per call from rayon workers / Python threads: examples/bench.rs:410-416, src/database/mod.rs:248-256;
    vdb_parallel_knn is that loop). Concurrent calls are coalesced into shared database passes by the library."""
    from lab_1806_vec_db_b200 import _lib as L
    lib = L.lib()
    out = {"k": k, "api": "vdb_flat_knn(nq=1, host pointers), one call per query from T native threads", "cases": []}
    ref = None
    for threads, nq in ((1, 256), (8, 2048), (32, 4096)):
        q = np.ascontiguousarray(q_host[:nq])
        ids = np.empty((nq, k), np.uint64); dd = np.empty((nq, k), np.float32); cnt = np.empty((nq,), np.uint32)
        secs = C.c_double(0)
        nb0, ns0 = C.c_uint64(0), C.c_uint64(0)
        lib.vdb_batch_stats(flat.vec_set._h, C.byref(nb0), C.byref(ns0))
        for _ in range(2):   # first round = warm-up
            L.check(lib.vdb_parallel_knn(flat.vec_set._h, L.ptr(q), nq, k, threads, L.ptr(ids), L.ptr(dd), L.ptr(cnt), C.byref(secs)))
        nb1, ns1 = C.c_uint64(0), C.c_uint64(0)
        lib.vdb_batch_stats(flat.vec_set._h, C.byref(nb1), C.byref(ns1))
        if ref is None:
            ref = (ids.copy(), dd.copy())
        m = min(nq, ref[0].shape[0])
        qps = nq / secs.value
        case = {"threads": threads, "calls": nq, "qps": qps,
                "queries_per_database_pass": (ns1.value - ns0.value) / max(1, nb1.value - nb0.value),
                "results_bit_identical_to_1_thread": bool((ids[:m] == ref[0][:m]).all() and
                                                          (dd[:m].view(np.uint32) == ref[1][:m].view(np.uint32)).all())}
        if threads == 1:
            case["ms_per_call"] = 1e3 / qps
            case["frac_of_hbm_peak_whole_call"] = n_rows * DIM * 4 * qps / 1e9 / peak_gbs
        else:
            case["speedup_vs_1_thread"] = qps / out["cases"][0]["qps"]
        out["cases"].append(case)
    return out


def run_reference(args):
    """--impl reference: the reference's CPU algorithm (oracle port) on the box's host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    nqs = args.cpu_queries or min(128, 2 * cores)
    base1000, test1000 = load_fixtures()
    try:
        import torch
        dev = torch.device("cuda:0") if torch.cuda.is_available() else torch.device("cpu")
    except Exception:
        dev = None
    import torch
    base = synth(base1000, 0, args.n, 42, dev).cpu().numpy()
    q = synth(test1000, 0, nqs, 43, dev).cpu().numpy()
    qps, dt, res = cpu_arm(base, q, args.k, cores, args.steps, min(args.warmup, 1))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *res)
    line = {
        "impl": "reference", "metric": "QPS, exact Flat L2 kNN", "value": qps, "unit": "queries/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        # the GPU arm's config (same workload, same keys); the bounded CPU sample is described under cpu_baseline
        "config": {"workload": f"Flat L2Sqr exact kNN, synthetic GIST-shaped {args.n}x{DIM} f32, "
                               f"{args.nq}-query batch, k={args.k} (configs[1])",
                   "n": args.n, "dim": DIM, "nq": args.nq, "k": args.k, "cpu_sample_queries_per_step": nqs},
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": cores, "kind": "port",
                         "sample": f"{nqs} of the {args.nq} queries x {args.n} rows per step, thread pool over queries "
                                   "(examples/bench.rs -t protocol); C++ restatement of the Rust path, "
                                   "sequential f32, -O3 -ffp-contract=off"},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_ours_multi(args):
    """N > 1: ONE process (rank 0) drives all N GPUs through the single C call a Rust host would make
    (vdb_flat_knn on a row-sharded handle: csrc/multi.cu - worker thread + stream per GPU, per-GPU top-k merged over
    NVLink peer memory). The driver launches one rank per GPU; ranks > 0 join the process group and the barriers and
    then measure the round-1 multi-process path (one shard per rank, NCCL all-gathers from Python: sharded.py) together
    with rank 0, reported beside the headline as `nccl_multiprocess`."""
    import torch
    import torch.distributed as dist
    import lab_1806_vec_db_b200 as V
    from lab_1806_vec_db_b200 import _lib as L
    from lab_1806_vec_db_b200.sharded import ShardedFlatIndex, shard_bounds

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    # host-side barrier group: while rank 0 drives every GPU, the other ranks must not park an NCCL kernel on "their"
    # GPU (two processes time-slice one GPU: a spinning barrier kernel of rank r would halve rank 0's share of GPU r)
    cpu_group = dist.new_group(backend="gloo")
    lib = L.lib()
    L.check(lib.vdb_set_device(local))
    path_code = {"auto": 0, "scan": 1, "tensor": 2}[args.path]
    L.check(lib.vdb_flat_set_path(path_code))
    base1000, test1000 = load_fixtures()

    def barrier():
        torch.cuda.synchronize()
        dist.barrier(group=cpu_group)

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- every rank: its own shard for the multi-process NCCL path (round-1 design, kept for comparison) ----
    lo, hi = shard_bounds(args.n, world, rank)
    base_r = synth(base1000, lo, hi, 42, dev)
    q_dev = synth(test1000, 0, args.nq, 43, dev)
    vs_r = V.DeviceVecSet.from_device(base_r.data_ptr(), hi - lo, DIM, DIM, np.float32, "l2sqr", id_base=lo, keepalive=base_r)
    idx_r = ShardedFlatIndex(vs_r, rank, world)
    q_pin = torch.empty((args.nq, DIM), dtype=torch.float32, pin_memory=True)
    q_pin.copy_(q_dev)
    out_pin = (torch.empty((args.nq, args.k), dtype=torch.int64, pin_memory=True),
               torch.empty((args.nq, args.k), dtype=torch.float32, pin_memory=True),
               torch.empty((args.nq,), dtype=torch.int32, pin_memory=True))

    # ---- rank 0: the single-process sharded handle over all N GPUs ----
    devs = list(range(world))
    if rank == 0:
        blocks, qd, bounds = [], [], []
        for s in devs:
            d = torch.device("cuda", s)
            b_lo, b_hi = shard_bounds(args.n, world, s)
            bounds.append((b_lo, b_hi))
            blocks.append(base_r if s == 0 else synth(base1000, b_lo, b_hi, 42, d))
            qd.append(q_dev if s == 0 else synth(test1000, 0, args.nq, 43, d))
        vs = V.DeviceVecSet.from_device_shards([b.data_ptr() for b in blocks], [b - a for a, b in bounds], devs, DIM, DIM,
                                               np.float32, "l2sqr", keepalive=blocks)
        flat = V.FlatIndex(vs)
        per = -(-args.nq // world)
        r_ids = [torch.empty((per, args.k), dtype=torch.int64, device=f"cuda:{s}") for s in devs]
        r_dd = [torch.empty((per, args.k), dtype=torch.float32, device=f"cuda:{s}") for s in devs]
        r_cnt = [torch.empty((per,), dtype=torch.int32, device=f"cuda:{s}") for s in devs]
        ptrs = lambda ts: [t.data_ptr() for t in ts]  # noqa: E731
        q_np = q_pin.numpy()
        out_np = (out_pin[0].numpy().view(np.uint64), out_pin[1].numpy(), out_pin[2].numpy().view(np.uint32))

        def dev_call():
            flat.knn_batch_sharded_dev(ptrs(qd), args.nq, args.k, ptrs(r_ids), ptrs(r_dd), ptrs(r_cnt))

        def sync_all():
            for s in devs:
                torch.cuda.synchronize(s)

        def events():
            evs = []
            for s in devs:
                with torch.cuda.device(s):
                    e = torch.cuda.Event(enable_timing=True)
                    e.record(torch.cuda.current_stream(s))
                    evs.append(e)
            return evs

    # ---- headline: device-resident, one C call per step on rank 0 (the other ranks wait at the barrier) ----
    ms = e2e_s = 0.0
    launches = 0
    clocks = None
    prof = {}
    if rank == 0:
        sampler = ClockSampler(0)
        sampler.wait_ready()
        for _ in range(args.warmup):
            dev_call()
        sync_all()
    barrier()
    if rank == 0:
        L.check(lib.vdb_prof_reset())
        L.check(lib.vdb_prof_enable(1))
        launches0 = lib.vdb_launch_count()
        sync_all()
        e0 = events()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            dev_call()                      # synchronous: every shard's stream has drained on return
        wall = time.perf_counter() - t0
        e1 = events()
        sync_all()
        ms = max(a.elapsed_time(b) for a, b in zip(e0, e1)) / args.steps
        launches = int(lib.vdb_launch_count() - launches0)
        L.check(lib.vdb_prof_enable(0))
        clocks = sampler.stop()
        for name in ("flat_scan", "flat_gemm", "flat_gemm_sample", "rerank", "merge", "mg_queries", "mg_sample", "mg_bcast", "mg_filter", "mg_finish", "mg_scatter", "mg_merge"):
            t, c = C.c_double(0), C.c_uint64(0)
            L.check(lib.vdb_prof_read(name.encode(), C.byref(t), C.byref(c)))
            prof[name] = (t.value, int(c.value))
        res = (torch.cat([t.cpu() for t in r_ids])[:args.nq].numpy(), torch.cat([t.cpu() for t in r_dd])[:args.nq].numpy(),
               torch.cat([t.cpu() for t in r_cnt])[:args.nq].numpy())
        stats = tensor_stats(lib)
    barrier()
    ms = max_over_ranks(ms)

    # ---- end to end: vdb_flat_knn with HOST buffers on the sharded handle (the call a Rust host makes) ----
    if rank == 0:
        flat.knn_batch(q_np, args.k, out_np)
    barrier()
    if rank == 0:
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_res = flat.knn_batch(q_np, args.k, out_np)
        e2e_s = (time.perf_counter() - t0) / args.steps
        e2e_same = bool((np.asarray(e2e_res[0]).view(np.int64) == res[0]).all())
    barrier()
    e2e_s = max_over_ranks(e2e_s)

    # ---- comparison: the multi-process path (one rank per GPU, NCCL all-gathers issued from Python) ----
    nccl = {}
    for _ in range(args.warmup):
        res_r = idx_r.knn_batch_dev(q_dev, args.k)
    barrier()
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a0.record()
    for _ in range(args.steps):
        res_r = idx_r.knn_batch_dev(q_dev, args.k)
    a1.record()
    barrier()
    nccl_ms = max_over_ranks(a0.elapsed_time(a1)) / args.steps
    idx_r.knn_batch(q_pin, args.k, out_pin)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        idx_r.knn_batch(q_pin, args.k, out_pin)
    barrier()
    nccl_e2e = max_over_ranks(time.perf_counter() - t0) / args.steps
    if rank != 0:
        dist.destroy_process_group()
        return
    nccl = {"value": args.nq / (nccl_ms * 1e-3), "ms_per_step": nccl_ms, "e2e_value": args.nq / nccl_e2e,
            "e2e_ms_per_step": nccl_e2e * 1e3, "ids_equal_single_process_result": bool((res_r[0].cpu().numpy() == res[0]).all()),
            "what": "round-1 path: one process per GPU (all N ranks), torch.distributed all-gathers between the vdb_tq_* phases"}

    # ---- roofline of the dominant kernel (per launch, averaged over the N GPUs) ----
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    n_local = bounds[0][1] - bounds[0][0]
    dom = max(("flat_scan", "flat_gemm"), key=lambda nm: prof[nm][0])
    t_dom, c_dom = prof[dom]
    if dom == "flat_scan":
        peak = peaks.get("hbm_gbs") or 6650.0
        per_launch = n_local * DIM * 4
        achieved = per_launch * c_dom / (t_dom * 1e-3) / 1e9 if t_dom > 0 else 0.0
        roof = {"bound": "hbm", "kernel": "flat_scan_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": None, "launches": c_dom, "avg_launch_ms": t_dom / max(c_dom, 1),
                "algorithmic_bytes_per_launch": per_launch, "scope": "per GPU"}
    else:
        flops = 2.0 * args.nq * n_local * DIM * args.steps * world     # all launches of all GPUs
        kind = C.c_int(-1)
        sh0 = C.c_void_p()
        L.check(lib.vdb_dataset_shard(vs._h, 0, C.byref(sh0), None, None, None))
        lib.vdb_dataset_operand_info(sh0, C.byref(kind), None, None, None, None)
        f16 = kind.value == 1
        peak, peak_src = tensor_peak(dev, peaks, f16)
        achieved = flops / (t_dom * 1e-3) / 1e12 if t_dom > 0 else 0.0  # t_dom sums the launches of all GPUs
        roof = {"bound": "tensor", "kernel": "flat_gemm_kernel", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                "frac": achieved / peak, "traffic": None, "scope": "per GPU (launch times summed over the GPUs)",
                "operand_kind": "f16 x f16 -> f32" if f16 else "tf32 x tf32 -> f32", "peak_source": peak_src,
                "launches": c_dom, "avg_launch_ms": t_dom / max(c_dom, 1), "flop_per_step_per_gpu": 2.0 * args.nq * n_local * DIM}
    roof["kernel_share_of_step"] = t_dom / world / (ms * args.steps) if ms > 0 else None

    # ---- parity of the sharded result against the CPU oracle (bounded query sample) ----
    cores = os.cpu_count() or 1
    nqs = args.cpu_queries or min(128, max(16, 4 * cores))
    base_host = np.empty((args.n, DIM), np.float32)
    for (b_lo, b_hi), blk in zip(bounds, blocks):
        base_host[b_lo:b_hi] = blk.cpu().numpy()
    q_host = q_pin[:nqs].numpy()
    qps_cpu, dt_cpu, ores = cpu_arm(base_host, q_host, args.k, cores, 1, 0)
    cpu = parity_fields(res, ores, q_host, base_host, nqs, args, cores, qps_cpu, dt_cpu)
    other = None
    if not args.no_other_configs:
        try:
            import bench_configs
            other = bench_configs.sharded_legs(V, vs, base_host, q_pin.numpy(), res[0][:, :10], world)
        except Exception as e:  # noqa: BLE001 - the headline line must not be lost to an auxiliary leg
            other = {"error": repr(e)}
    del base_host

    line = {
        "metric": "QPS, exact Flat L2 kNN", "value": args.nq / (ms * 1e-3), "unit": "queries/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"Flat L2Sqr exact kNN, synthetic GIST-shaped {args.n}x{DIM} f32, "
                               f"{args.nq}-query batch, k={args.k} (configs[1])",
                   "n": args.n, "dim": DIM, "nq": args.nq, "k": args.k, "path": args.path,
                   "sharding": f"rows in {world} contiguous block(s), one per GPU; ONE process drives all GPUs through one "
                               "C call (vdb_flat_knn_sharded_dev / vdb_flat_knn), per-GPU top-k merged over NVLink peer memory",
                   "l2_policy": "inputs (3.84 GB per pass) larger than the 126 MB L2"},
        "e2e": {"value": args.nq / e2e_s, "unit": "queries/s", "h2d_bytes_per_step": args.nq * DIM * 4,
                "d2h_bytes_per_step": args.nq * args.k * 12 + args.nq * 4, "ms_per_step": e2e_s * 1e3,
                "api": "vdb_flat_knn (host pointers) on the row-sharded handle: every GPU uploads 1/N of the batch over its "
                       "own PCIe link, broadcasts it over NVLink, and downloads the slice of the results it owns",
                "host_buffers": "page-locked, reused across steps", "ids_equal_device_resident_result": e2e_same},
        "gpu_launches": launches, "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
        "kernel_ms": {k_: {"ms": v[0], "launches": v[1]} for k_, v in prof.items()},
        "tensor_path": stats, "host_wall_ms_per_step": wall / args.steps * 1e3, "nccl_multiprocess": nccl,
        "other_configs": other,
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *res)
    print(json.dumps(line), flush=True)
    dist.destroy_process_group()


def parity_fields(res, ores, q_host, base_host, nqs, args, cores, qps_cpu, dt_cpu):
    """cpu_baseline object: the oracle's throughput on the bounded sample + the parity spot check of the GPU result."""
    import oracle as O
    ids_gpu = np.asarray(res[0][:nqs]).astype(np.int64)
    match = float((ids_gpu == ores[0].astype(np.int64)).mean())
    dd_gpu = np.asarray(res[1][:nqs])
    rel = float(np.max(np.abs(dd_gpu - ores[1]) / np.maximum(np.abs(ores[1]), 1e-6)))
    # every id mismatch must be a tie within 1e-5 relative distance (the parity rule of BASELINE.json)
    ties_ok = True
    for qi, j in zip(*np.nonzero(ids_gpu != ores[0].astype(np.int64))):
        d = O.distance(q_host[qi], base_host[int(ids_gpu[qi, j])], "l2sqr")
        ties_ok &= abs(d - ores[1][qi, j]) <= 1e-5 * abs(ores[1][qi, j]) + 1e-6
    return {"value": qps_cpu, "unit": "queries/s", "cores": cores, "kind": "port",
            "sample": f"{nqs} of the {args.nq} queries x {args.n} rows, one pass, thread pool over queries; "
                      "oracle = C++ restatement of the Rust path (sequential f32, no FMA)",
            "seconds": dt_cpu, "gpu_vs_cpu_exact_id_rate": match, "gpu_vs_cpu_max_rel_dist_err": rel,
            "id_mismatches_are_ties_within_1e-5": bool(ties_ok)}


def run_ours(args):
    import torch
    import torch.distributed as dist
    import lab_1806_vec_db_b200 as V
    from lab_1806_vec_db_b200 import _lib as L
    from lab_1806_vec_db_b200.sharded import ShardedFlatIndex, shard_bounds

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = L.lib()
    L.check(lib.vdb_set_device(local))
    L.check(lib.vdb_flat_set_path({"auto": 0, "scan": 1, "tensor": 2}[args.path]))

    base1000, test1000 = load_fixtures()
    lo, hi = shard_bounds(args.n, world, rank)
    base = synth(base1000, lo, hi, 42, dev)
    q_dev = synth(test1000, 0, args.nq, 43, dev)
    vs = V.DeviceVecSet.from_device(base.data_ptr(), hi - lo, DIM, DIM, np.float32, "l2sqr", id_base=lo,
                                    keepalive=base)
    idx = ShardedFlatIndex(vs, rank, world)
    flat = V.FlatIndex(vs)
    q_pin = torch.empty((args.nq, DIM), dtype=torch.float32, pin_memory=True)
    q_pin.copy_(q_dev)
    out_pin = (torch.empty((args.nq, args.k), dtype=torch.int64, pin_memory=True),
               torch.empty((args.nq, args.k), dtype=torch.float32, pin_memory=True),
               torch.empty((args.nq,), dtype=torch.int32, pin_memory=True))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident timing (value) -----------------------------------------------------------
    res = None
    sampler = ClockSampler(local) if rank == 0 else None  # started early: nvidia-smi needs ~0.3 s to emit samples
    if sampler:
        sampler.wait_ready()
    for _ in range(args.warmup):
        res = idx.knn_batch_dev(q_dev, args.k)
    barrier()
    L.check(lib.vdb_prof_reset())
    L.check(lib.vdb_prof_enable(1))
    launches0 = lib.vdb_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        res = idx.knn_batch_dev(q_dev, args.k)
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1)) / args.steps
    launches = int(lib.vdb_launch_count() - launches0)
    L.check(lib.vdb_prof_enable(0))
    clocks = sampler.stop() if sampler else None

    prof = {}
    for name in ("flat_scan", "flat_gemm", "flat_gemm_sample", "rerank", "merge"):
        t, c = C.c_double(0), C.c_uint64(0)
        L.check(lib.vdb_prof_read(name.encode(), C.byref(t), C.byref(c)))
        prof[name] = (t.value, int(c.value))

    # the same contraction kernel timed ALONE (VDB_GEMM_PARTS=1: one filter launch per step, the rerank strictly
    # after it). In the timed region above the filter pass is cut into row parts and the rerank gathers of part i run
    # on a side stream under the launch of part i + 1: the step is shorter, each launch is longer.
    alone = None
    if rank == 0 and world == 1 and args.path != "scan" and int(os.environ.get("VDB_GEMM_PARTS", "1")) > 1:
        keep = os.environ.get("VDB_GEMM_PARTS")
        os.environ["VDB_GEMM_PARTS"] = "1"
        idx.knn_batch_dev(q_dev, args.k)
        torch.cuda.synchronize()
        L.check(lib.vdb_prof_reset())
        L.check(lib.vdb_prof_enable(1))
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(3):
            idx.knn_batch_dev(q_dev, args.k)
        a1.record()
        torch.cuda.synchronize()
        L.check(lib.vdb_prof_enable(0))
        t, c = C.c_double(0), C.c_uint64(0)
        L.check(lib.vdb_prof_read(b"flat_gemm", C.byref(t), C.byref(c)))
        alone = {"flat_gemm_ms_per_step": t.value / 3, "launches_per_step": int(c.value) // 3,
                 "ms_per_step": a0.elapsed_time(a1) / 3}
        if keep is None:
            del os.environ["VDB_GEMM_PARTS"]
        else:
            os.environ["VDB_GEMM_PARTS"] = keep

    # ---- end-to-end timing through the host-buffer API (e2e) --------------------------------------
    q_np = q_pin.numpy()
    # caller-owned, page-locked result arrays reused across the steps (a Rust caller reuses its Vecs the same way)
    out_np = (out_pin[0].numpy().view(np.uint64), out_pin[1].numpy(), out_pin[2].numpy().view(np.uint32))
    def e2e_call():
        if world == 1:
            return flat.knn_batch(q_np, args.k, out_np)  # the C-ABI call a Rust caller makes (vdb_flat_knn)
        return idx.knn_batch(q_pin, args.k, out_pin)
    e2e_call()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_res = e2e_call()
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0) / args.steps

    # the end-to-end call must return what the device-resident call returned
    e2e_ids = np.asarray(e2e_res[0]).view(np.int64) if world == 1 else e2e_res[0].numpy()
    e2e_same = bool((e2e_ids == res[0].cpu().numpy()).all())

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel ------------------------------------------------------------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    n_local = hi - lo
    dom = max(("flat_scan", "flat_gemm"), key=lambda nm: prof[nm][0])
    t_dom, c_dom = prof[dom]
    if dom == "flat_scan":
        peak, src = (peaks.get("hbm_gbs"), "measured") if peaks.get("hbm_gbs") else (6650.0, "fallback")
        per_launch = n_local * DIM * 4  # algorithmic bytes of one database pass (DESIGN.md K1)
        achieved = per_launch * c_dom / (t_dom * 1e-3) / 1e9 if t_dom > 0 else 0.0
        roof = {"bound": "hbm", "kernel": "flat_scan_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": None, "peak_source": src,
                "launches": c_dom, "avg_launch_ms": t_dom / max(c_dom, 1),
                "algorithmic_bytes_per_launch": per_launch}
    else:
        # dense contraction: 2*nq*n*dim FLOP per step = the filter launches; the sample passes (ns/n ~ 3 % more FLOP) are
        # timed under their own name ("flat_gemm_sample" in kernel_ms) and counted in neither numerator nor denominator
        flops = 2.0 * args.nq * n_local * DIM * args.steps
        tstats = tensor_stats(lib, vs._h) or {}
        f16 = "fp16" in (tstats.get("operand") or {}).get("kind", "")
        peak, peak_src = tensor_peak(dev, peaks, f16)
        achieved = flops / (t_dom * 1e-3) / 1e12 if t_dom > 0 else 0.0
        roof = {"bound": "tensor", "kernel": "flat_gemm_kernel", "achieved": achieved, "peak": peak,
                "unit": "TFLOP/s", "frac": achieved / peak,
                "operand_kind": "f16 x f16 -> f32 (tcgen05.mma.kind::f16)" if f16 else "tf32 x tf32 -> f32 (tcgen05.mma.kind::tf32)",
                # dram__bytes_read.sum + dram__bytes_write.sum of one filter launch from the committed ncu capture
                "traffic": (GEMM_PASS_TRAFFIC if (n_local == 1_000_000 and args.nq == 10_000 and f16 and
                                                  int(os.environ.get("VDB_GEMM_PARTS", "1")) == 1) else None),
                "traffic_source": "ncu --set full capture of this launch, profiles/r02_flat_gemm_ncu.md (a constant from that "
                                  "capture, not measured in this run)",
                "algorithmic_bytes_per_launch": n_local * (DIM * (2 if f16 else 4) + 12) + args.nq * DIM * (2 if f16 else 4),
                "peak_source": peak_src,
                "launches": c_dom, "avg_launch_ms": t_dom / max(c_dom, 1),
                "flop_per_step": flops / args.steps}
    roof["kernel_share_of_step"] = t_dom / (ms * args.steps) if ms > 0 else None
    if dom == "flat_gemm" and alone:
        a_ach = 2.0 * args.nq * n_local * DIM / (alone["flat_gemm_ms_per_step"] * 1e-3) / 1e12
        roof["note"] = ("achieved/frac are over the timed region, where the filter launches share the GPU with the "
                        "rerank gathers of the previous row part (side stream); `alone` is the same kernel with "
                        "VDB_GEMM_PARTS=1 (nothing concurrent), 3 extra steps after the timed region")
        roof["alone"] = {"achieved": a_ach, "frac": a_ach / roof["peak"], **alone}

    # ---- CPU baseline (bounded sample) + parity spot check -----------------------------------------
    cpu = None
    if world == 1:
        cores = os.cpu_count() or 1
        nqs = args.cpu_queries or min(128, max(16, 4 * cores))  # ~2.5 s of wall clock = ~40 core-seconds per pass
        base_host = base.cpu().numpy()
        q_host = q_pin[:nqs].numpy()
        qps_cpu, dt_cpu, ores = cpu_arm(base_host, q_host, args.k, cores, 1, 0)
        cpu = parity_fields((res[0].cpu().numpy(), res[1].cpu().numpy()), ores, q_host, base_host, nqs, args, cores, qps_cpu, dt_cpu)
        del base_host

    # ---- the HBM-bound regime of the same path: the trait's small-batch call through the streaming scan (K1) ----
    hbm_scan = None
    if world == 1:
        peak_hbm = peaks.get("hbm_gbs") or 6650.0
        hbm_scan = {"kernel": "flat_scan_kernel", "peak_gbs": peak_hbm,
                    "peak_source": "measured" if peaks.get("hbm_gbs") else "fallback", "k": 10, "cases": []}
        L.check(lib.vdb_flat_set_path(1))
        for nq1 in (1, 2, 4, 8):
            qs = q_dev[:nq1].contiguous()
            for _ in range(40 if nq1 == 1 else 3):  # the first case also brings the clocks back up after the CPU leg
                idx.knn_batch_dev(qs, 10)
            # whole call first, WITHOUT the library's per-kernel events (they add launch gaps), then the kernel alone
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 50
            a0.record()
            for _ in range(reps):
                idx.knn_batch_dev(qs, 10)
            a1.record()
            torch.cuda.synchronize()
            call_ms = a0.elapsed_time(a1) / reps
            L.check(lib.vdb_prof_reset())
            L.check(lib.vdb_prof_enable(1))
            for _ in range(20):
                idx.knn_batch_dev(qs, 10)
            torch.cuda.synchronize()
            L.check(lib.vdb_prof_enable(0))
            t, c = C.c_double(0), C.c_uint64(0)
            L.check(lib.vdb_prof_read(b"flat_scan", C.byref(t), C.byref(c)))
            kern_ms = t.value / max(int(c.value), 1)
            gbs = n_local * DIM * 4 / (kern_ms * 1e-3) / 1e9
            hbm_scan["cases"].append({"nq": nq1, "qps": nq1 / (call_ms * 1e-3), "call_ms": call_ms,
                                      "scan_kernel_ms": kern_ms, "achieved_gbs": gbs, "frac": gbs / peak_hbm,
                                      "frac_whole_call": n_local * DIM * 4 / (call_ms * 1e-3) / 1e9 / peak_hbm})
        L.check(lib.vdb_flat_set_path({"auto": 0, "scan": 1, "tensor": 2}[args.path]))
        # the same small batches through the AUTO path (what a caller gets): from 3 queries up the library answers with
        # one single-CTA tensor pass over the 2-byte operand copy (half the bytes of the f32 rows) + exact rerank
        hbm_scan["auto_path"] = []
        for nq1 in (2, 3, 4, 8, 32, 128):
            qs = q_dev[:nq1].contiguous()
            for _ in range(3):
                idx.knn_batch_dev(qs, 10)
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 20
            a0.record()
            for _ in range(reps):
                idx.knn_batch_dev(qs, 10)
            a1.record()
            torch.cuda.synchronize()
            call_ms = a0.elapsed_time(a1) / reps
            hbm_scan["auto_path"].append({"nq": nq1, "qps": nq1 / (call_ms * 1e-3), "call_ms": call_ms,
                                          "f32_row_bytes_per_call_over_peak": n_local * DIM * 4 / (call_ms * 1e-3) / 1e9 / peak_hbm})

    # ---- the reference's real call pattern: ONE query per knn call, host pointers, from 1 / 8 / 32 caller threads ----
    single = None
    if world == 1:
        single = single_query_e2e(flat, q_pin.numpy(), n_local, peaks.get("hbm_gbs") or 6650.0)

    # ---- the other single-GPU configs of BASELINE.json on the same rows (IVF, PQ) ----------------------------
    other = None
    if world == 1 and not args.no_other_configs and args.n >= 65536:
        try:
            import bench_configs
            other = bench_configs.run_all(V, L, lib, dev, peaks, base, q_dev, synth_clustered, base1000, args.n)
        except Exception as e:  # the headline line must not be lost to an auxiliary leg
            other = {"error": repr(e)}

    qps = args.nq / (ms * 1e-3)
    line = {
        "metric": "QPS, exact Flat L2 kNN", "value": qps, "unit": "queries/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"Flat L2Sqr exact kNN, synthetic GIST-shaped {args.n}x{DIM} f32, "
                               f"{args.nq}-query batch, k={args.k} (configs[1])",
                   "n": args.n, "dim": DIM, "nq": args.nq, "k": args.k, "path": args.path,
                   "sharding": f"rows in {world} contiguous block(s), one per GPU",
                   "l2_policy": "inputs (3.84 GB per pass) larger than the 126 MB L2"},
        "e2e": {"value": args.nq / e2e_s, "unit": "queries/s", "h2d_bytes_per_step": args.nq * DIM * 4,
                "d2h_bytes_per_step": args.nq * args.k * 12 + args.nq * 4, "ms_per_step": e2e_s * 1e3,
                "api": "vdb_flat_knn (host pointers)" if world == 1 else "ShardedFlatIndex.knn_batch (pinned host)",
                "host_buffers": "page-locked, reused across steps", "ids_equal_device_resident_result": e2e_same},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": roof,
        "cpu_baseline": cpu,
        "kernel_ms": {k_: {"ms": v[0], "launches": v[1]} for k_, v in prof.items()},
        "tensor_path": tensor_stats(lib, vs._h),
        "hbm_scan": hbm_scan,
        "e2e_single_query": single,
        "other_configs": other,
    }
    if idx.phase_ms.get("calls"):  # VDB_PHASE_TIMING=1: per-phase device time of the sharded search (rank 0), ms per call
        line["phase_ms"] = {k_: round(v / idx.phase_ms["calls"], 4) for k_, v in idx.phase_ms.items() if k_ != "calls"}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *(t.cpu().numpy() for t in res))
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    elif int(os.environ.get("WORLD_SIZE", "1")) > 1:
        run_ours_multi(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
