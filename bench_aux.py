#!/usr/bin/env python
"""bench_aux.py — the other 1M x 960 configs of BASELINE.json (not the headline line of bench.py):

  C3  IVF  nlist=128, k-means on a 100k-row sample (20 iters), nprobe in {8,12,16,20,24}, k=10
           (config/bench_10000_ivf.toml scaled x100)
  C4  PQ   m=240, 4 bits, k-means on 10k rows (20 iters), Flat+PQ scan, ef in {240..600 step 60}, k=10
           (config/bench_pq_240_hnsw.toml:16-23, examples/bench.rs protocol: recall@10 vs Flat ground truth)

  ivfpq  IVF + PQ (IVFIndex.knn_pq): the C3 lists and the C4 table, nprobe in {8,16,32} x ef in {60,120,240}, at nq =
           1000 and nq = 1, next to IVF knn_with_ef and Flat knn_pq at the same settings, with the ADC lookups of the
           scan and their floor (32 shared-memory reads per clock per SM)

Prints one JSON line per measurement. 1000 queries (as examples/bench.rs), synthetic GIST-shaped data of bench.py
(--data clustered: bench.synth_clustered, where PQ / IVF recall is meaningful).
The CPU column is the oracle (reference semantics) on a bounded query sample.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
from bench import DIM, load_fixtures, synth, synth_clustered  # noqa: E402


def timed(fn, reps=3):
    import torch
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, out


def recall_at(ids, gt):
    hit = 0
    for a, b in zip(ids, gt):
        hit += len(set(a.tolist()) & set(b.tolist()))
    return hit / gt.size


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--nq", type=int, default=1000)
    ap.add_argument("--what", default="ivf,pq")
    ap.add_argument("--hnsw-m", type=int, default=16)
    ap.add_argument("--hnsw-efc", type=int, default=200)
    ap.add_argument("--hnsw-ef", default="120:360:40", help="start:end:step of the HNSW ef sweep")
    ap.add_argument("--hnsw-cpu", action="store_true", help="also build / search the CPU restatement (small n only)")
    ap.add_argument("--hnsw-pq", action="store_true", help="also HNSW + PQ (config/bench_pq_240_hnsw.toml): knn_pq on the graph")
    ap.add_argument("--cpu-queries", type=int, default=8)
    ap.add_argument("--pq-m", type=int, default=240)
    ap.add_argument("--ef", default="240:600:60", help="start:end:step of the PQ ef sweep")
    ap.add_argument("--data", choices=("synth", "clustered"), default="synth")
    args = ap.parse_args()
    what = set(args.what.split(","))
    import torch
    import lab_1806_vec_db_b200 as V
    from lab_1806_vec_db_b200 import _lib as L
    import oracle as O

    dev = torch.device("cuda:0")
    lib = L.lib()
    base1000, test1000 = load_fixtures()
    gen = synth_clustered if args.data == "clustered" else synth
    base = gen(base1000, 0, args.n, 42, dev)
    q_dev = gen(test1000, 0, args.nq, 43, dev)
    vs = V.DeviceVecSet.from_device(base.data_ptr(), args.n, DIM, DIM, np.float32, "l2sqr", keepalive=base)
    flat = V.FlatIndex(vs)
    base_host = base.cpu().numpy()
    q_host = q_dev.cpu().numpy()
    cores = os.cpu_count() or 1
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    k = 10
    gt_ids, _, _ = flat.knn_batch(q_host, k)  # exact ground truth (gen_gnd.rs protocol)
    gt_ids = gt_ids.astype(np.int64)
    rng = np.random.default_rng(42)

    def dev_out():
        return (torch.empty((args.nq, k), dtype=torch.int64, device=dev),
                torch.empty((args.nq, k), dtype=torch.float32, device=dev),
                torch.empty((args.nq,), dtype=torch.int32, device=dev))

    def build_ivf():
        t0 = time.perf_counter()
        train = np.ascontiguousarray(base_host[rng.permutation(args.n)[:min(100_000, args.n)]])
        km = V.KMeans.from_vec_set(train, V.KMeansConfig(128, 20, 1e-6, "l2sqr"), rng)
        t_train = time.perf_counter() - t0
        t0 = time.perf_counter()
        ivf = V.IVFIndex(vs, km.centroids)
        t_assign = time.perf_counter() - t0
        sizes = np.array([len(c) for c in ivf.clusters])
        # CPU: assignment on a row sample (ivf_index.rs:89-93), probe scan on a query sample
        ns = 20_000
        t0 = time.perf_counter()
        a_cpu = O.kmeans_assign(base_host[:ns], km.centroids, "l2sqr", nthreads=cores)
        cpu_assign_s = (time.perf_counter() - t0) * args.n / ns
        assert (a_cpu == ivf.assignment[:ns]).all(), "IVF assignment differs from the oracle"
        off, mem = O.ivf_lists(ivf.assignment, 128)
        return km, ivf, sizes, off, mem, t_train, t_assign, cpu_assign_s, ns

    if "ivf" in what:
        km, ivf, sizes, off, mem, t_train, t_assign, cpu_assign_s, ns = build_ivf()
        print(json.dumps({"config": "C3 IVF build", "n": args.n, "nlist": 128, "kmeans_iters": km.iterations,
                          "gpu_train_s": t_train, "gpu_assign_lists_s": t_assign,
                          "cpu_assign_s_extrapolated": cpu_assign_s, "cpu_cores": cores,
                          "list_min_max": [int(sizes.min()), int(sizes.max())],
                          "assignment_bit_exact_vs_oracle_on_rows": ns}), flush=True)
        for nprobe in (8, 12, 16, 20, 24):
            ids, dd, cnt = dev_out()

            def run():
                L.check(lib.vdb_ivf_knn_dev(vs._h, ivf._h, C.c_void_p(q_dev.data_ptr()), args.nq, k, nprobe,
                                            C.c_void_p(ids.data_ptr()), C.c_void_p(dd.data_ptr()),
                                            C.c_void_p(cnt.data_ptr()), st))
            ms, _ = timed(run)
            rec = recall_at(ids.cpu().numpy(), gt_ids)
            nc = args.cpu_queries
            t0 = time.perf_counter()
            oi, od, oc = O.ivf_knn(base_host, km.centroids, off, mem, q_host[:nc], k, nprobe, "l2sqr", nthreads=cores)
            cpu_qps = nc / (time.perf_counter() - t0)
            same = float((ids[:nc].cpu().numpy() == oi.astype(np.int64)).mean())
            visited = float(np.mean([sum(sizes[c] for c in O.find_n_nearest(q_host[i], km.centroids, nprobe, "l2sqr"))
                                     for i in range(min(32, args.nq))]))
            gbs = visited * DIM * 4 * args.nq / (ms * 1e-3) / 1e9
            print(json.dumps({"config": "C3 IVF search", "nprobe": nprobe, "k": k, "nq": args.nq, "qps": args.nq / ms * 1e3,
                              "ms_per_batch": ms, "recall@10": rec, "rows_visited_per_query": visited,
                              "achieved_gbs": gbs, "hbm_frac_of_6551": gbs / 6551.4, "cpu_qps": cpu_qps,
                              "cpu_cores": cores, "cpu_queries": nc, "gpu_vs_oracle_exact_id_rate": same}), flush=True)

    def build_pq():
        t0 = time.perf_counter()
        M = args.pq_m
        cfg = V.PQConfig(4, M, "l2sqr", min(10_000, args.n), 20, 1e-6)
        train = np.ascontiguousarray(base_host[rng.permutation(args.n)[:min(10_000, args.n)]])
        from lab_1806_vec_db_b200.index import train_codebooks
        train_dev = V.DeviceVecSet(train, "l2sqr")
        t1 = time.perf_counter()
        books = train_codebooks(train_dev, cfg, rng)          # all m groups in one launch (vdb_pq_train_ds)
        t_kernel = time.perf_counter() - t1
        train_dev.close()
        t_train = time.perf_counter() - t0
        print(json.dumps({"config": "C4 PQ train", "m": M, "rows": len(train), "gpu_train_s_incl_upload": t_train,
                          "gpu_train_call_s": t_kernel,
                          "iterations_min_max": [int(train_codebooks.last_iterations.min()),
                                                 int(train_codebooks.last_iterations.max())]}), flush=True)
        t0 = time.perf_counter()
        pq = V.PQTable(vs, cfg, books)
        return M, books, pq, t_train, time.perf_counter() - t0

    if "pq" in what:
        M, books, pq, t_train, t_encode = build_pq()
        ns = 2000
        t0 = time.perf_counter()
        c_cpu = O.pq_encode(base_host[:ns], books, M, 4, "l2sqr", nthreads=1)  # the reference encodes serially
        cpu_encode_s = (time.perf_counter() - t0) * args.n / ns
        assert (c_cpu == pq.encoded_vec_set[:ns]).all(), "PQ codes differ from the oracle"
        print(json.dumps({"config": "C4 PQ build", "n": args.n, "m": M, "n_bits": 4, "gpu_train_s": t_train,
                          "gpu_encode_s_incl_d2h": t_encode, "cpu_encode_s_extrapolated_1_thread": cpu_encode_s,
                          "codes_bit_exact_vs_oracle_on_rows": ns}), flush=True)
        e0, e1, es = (int(x) for x in args.ef.split(":"))
        for ef in range(e0, e1 + 1, es):
            ids, dd, cnt = dev_out()

            def run():
                L.check(lib.vdb_pq_knn_dev(vs._h, pq._h, C.c_void_p(q_dev.data_ptr()), args.nq, k, ef,
                                           C.c_void_p(ids.data_ptr()), C.c_void_p(dd.data_ptr()),
                                           C.c_void_p(cnt.data_ptr()), st))
            ms, _ = timed(run)
            rec = recall_at(ids.cpu().numpy(), gt_ids)
            nc = args.cpu_queries
            t0 = time.perf_counter()
            oi, od, oc = O.flat_knn_pq(base_host, pq.encoded_vec_set, books, M, 4, q_host[:nc], k, ef, "l2sqr",
                                       nthreads=cores)
            cpu_qps = nc / (time.perf_counter() - t0)
            same = float((ids[:nc].cpu().numpy() == oi.astype(np.int64)).mean())
            gbs = args.n * ((M + 1) // 2) * ((args.nq + 3) // 4) / (ms * 1e-3) / 1e9
            print(json.dumps({"config": "C4 Flat+PQ search", "ef": ef, "k": k, "nq": args.nq, "qps": args.nq / ms * 1e3,
                              "ms_per_batch": ms, "recall@10": rec, "code_bytes_per_pass": args.n * ((M + 1) // 2),
                              "achieved_code_gbs": gbs, "cpu_qps": cpu_qps, "cpu_cores": cores, "cpu_queries": nc,
                              "gpu_vs_oracle_exact_id_rate": same}), flush=True)

    if "hnsw" in what:
        # C5: config/bench_hnsw.toml (M = 16 default, ef_construction = 200, ef 120..360 step 40, k = 10)
        L.check(lib.vdb_prof_reset())
        L.check(lib.vdb_prof_enable(1))
        t0 = time.perf_counter()
        hn = V.HNSWIndex(vs, V.HNSWConfig(0, args.hnsw_efc, args.hnsw_m), rng=np.random.default_rng(42))
        t_build = time.perf_counter() - t0
        L.check(lib.vdb_prof_enable(0))
        kern = {}
        for name in (b"hnsw_search", b"hnsw_select", b"hnsw_arrange"):
            t, c = C.c_double(0), C.c_uint64(0)
            L.check(lib.vdb_prof_read(name, C.byref(t), C.byref(c)))
            kern[name.decode()] = {"s": t.value / 1e3, "launches": c.value}
        links, lens = hn.level0_links()
        print(json.dumps({"config": "C5 HNSW build", "n": args.n, "M": args.hnsw_m, "ef_construction": args.hnsw_efc,
                          "gpu_build_s": t_build, "inserts_per_s": args.n / t_build, "kernels": kern,
                          "level0_degree_mean": float(lens.mean()), "level0_degree_max": int(lens.max()),
                          "enter": hn.enter_point, "max_batch": V.HNSWIndex.MAX_BATCH}), flush=True)
        ref = None
        if args.hnsw_cpu:
            from oracle.oracle_py import HnswOracle
            t0 = time.perf_counter()
            ref = HnswOracle(base_host, "l2sqr", args.hnsw_m, args.hnsw_efc, hn.levels)   # same levels, one thread
            print(json.dumps({"config": "C5 HNSW build (CPU restatement, 1 thread)", "n": args.n,
                              "cpu_build_s": time.perf_counter() - t0}), flush=True)
        e0, e1, es = (int(x) for x in args.hnsw_ef.split(":"))
        if os.environ.get("VDB_CUPROF"):   # ncu --profile-from-start off: capture the SEARCH launches, not the build's
            torch.cuda.cudart().cudaProfilerStart()
        for ef in range(e0, e1 + 1, es):
            ids, dd, cnt = dev_out()
            if ref is not None:
                t0 = time.perf_counter()
                oi, _, _ = ref.knn(q_host, k, ef, nthreads=cores)
                cpu_s = time.perf_counter() - t0
                print(json.dumps({"config": "C5 HNSW search (CPU restatement)", "ef": ef, "cpu_qps": args.nq / cpu_s,
                                  "cpu_cores": cores, "recall@10": recall_at(oi.astype(np.int64), gt_ids)}), flush=True)

            def run():
                L.check(lib.vdb_hnsw_knn_dev(vs._h, hn._h, C.c_void_p(q_dev.data_ptr()), args.nq, k, ef,
                                             C.c_void_p(ids.data_ptr()), C.c_void_p(dd.data_ptr()),
                                             C.c_void_p(cnt.data_ptr()), st))
            ms, _ = timed(run)
            rec = recall_at(ids.cpu().numpy(), gt_ids)
            print(json.dumps({"config": "C5 HNSW search", "ef": ef, "k": k, "nq": args.nq, "qps": args.nq / ms * 1e3,
                              "ms_per_batch": ms, "recall@10": rec}), flush=True)
        if args.hnsw_pq:
            M, books, pq, t_train, t_encode = build_pq()
            e0, e1, es = (int(x) for x in args.ef.split(":"))
            for ef in range(e0, e1 + 1, es):
                ids, dd, cnt = dev_out()

                def run():
                    L.check(lib.vdb_hnsw_knn_pq_dev(vs._h, hn._h, pq._h, C.c_void_p(q_dev.data_ptr()), args.nq, k, ef,
                                                    C.c_void_p(ids.data_ptr()), C.c_void_p(dd.data_ptr()),
                                                    C.c_void_p(cnt.data_ptr()), st))
                ms, _ = timed(run)
                rec = recall_at(ids.cpu().numpy(), gt_ids)
                print(json.dumps({"config": "C5 HNSW+PQ search", "m": M, "ef": ef, "k": k, "nq": args.nq,
                                  "qps": args.nq / ms * 1e3, "ms_per_batch": ms, "recall@10": rec}), flush=True)

    if "ivfpq" in what:
        ivfpq_sweep(args, V, L, O, lib, vs, flat, q_dev, q_host, base_host, gt_ids, st, dev_out, build_ivf, build_pq, k, cores)


def card_info():
    """Card name, power limit and maximum SM clock, read in the same run as the measurement."""
    import torch
    info = {"card": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["max_sm_clock_mhz"] = float(out[0]), float(out[1])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        info["power_limit_w"] = info["max_sm_clock_mhz"] = None
    return info


def ivfpq_sweep(args, V, L, O, lib, vs, flat, q_dev, q_host, base_host, gt_ids, st, dev_out, build_ivf, build_pq, k, cores):
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from ivf_pq_reference import ivf_knn_pq   # the oracle-composed IVF knn_pq reference of the tests
    card = card_info()
    km, ivf, sizes, off, mem, *_ = build_ivf()
    M, books, pq, _, _ = build_pq()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    clock_hz = (card["max_sm_clock_mhz"] or 1965.0) * 1e6
    probes = {p: [O.find_n_nearest(q_host[i], km.centroids, p, "l2sqr") for i in range(args.nq)] for p in (8, 16, 32)}

    def kernel_ms(run, name):
        L.check(lib.vdb_prof_reset())
        L.check(lib.vdb_prof_enable(1))
        run()
        L.check(lib.vdb_prof_enable(0))
        t, c = C.c_double(0), C.c_uint64(0)
        L.check(lib.vdb_prof_read(name, C.byref(t), C.byref(c)))
        return t.value

    for nq in (args.nq, 1):
        ids, dd, cnt = dev_out()
        reps = 3 if nq > 1 else 1

        def timed_calls(call):
            """ms per batch of nq queries (nq = 1: 200 single-query calls, each ending in its device synchronise)"""
            if nq > 1:
                return timed(lambda: call(q_dev, nq, ids, dd, cnt), reps)[0]
            call(q_dev, 1, ids, dd, cnt)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(200):
                call(q_dev[i], 1, ids[i], dd[i], cnt[i])
            torch.cuda.synchronize()
            return (time.perf_counter() - t0) * 1e3 / 200

        def p(t):
            return C.c_void_p(t.data_ptr())
        nrec = args.nq if nq > 1 else 200
        for nprobe in (8, 16, 32):
            ms_ivf = timed_calls(lambda q, n, i, d, c: L.check(lib.vdb_ivf_knn_dev(vs._h, ivf._h, p(q), n, k, nprobe, p(i), p(d), p(c), st)))
            rec_ivf = recall_at(ids[:nrec].cpu().numpy(), gt_ids[:nrec])
            print(json.dumps({"config": "IVF knn_with_ef (same nprobe)", "nq": nq, "nprobe": nprobe, "qps": nq / ms_ivf * 1e3,
                              "ms_per_batch": ms_ivf, "recall@10": rec_ivf, **card}), flush=True)
            visited = np.array([sum(int(sizes[c]) for c in probes[nprobe][i]) for i in range(args.nq)])
            for ef in (60, 120, 240):
                def call(q, n, i, d, c):
                    L.check(lib.vdb_ivf_knn_pq_dev(vs._h, ivf._h, pq._h, p(q), n, k, ef, nprobe, p(i), p(d), p(c), st))
                ms = timed_calls(call)
                got = ids[:nrec].cpu().numpy()
                rec = recall_at(got, gt_ids[:nrec])
                scan_ms = kernel_ms(lambda: call(q_dev, nq, ids, dd, cnt), b"ivf_pq_scan")
                lookups = float(visited[:nq].sum()) * M
                floor_ms = lookups / (sms * 32 * clock_hz) * 1e3
                nc = min(args.cpu_queries, nq)
                (oi, _, _), _ = ivf_knn_pq(O, base_host, pq.encoded_vec_set, books, M, 4, km.centroids, off, mem, q_host[:nc],
                                           k, ef, nprobe, "l2sqr")
                same = float((got[:nc] == oi.astype(np.int64)).mean())
                print(json.dumps({"config": "IVF+PQ knn_pq", "nq": nq, "nprobe": nprobe, "ef": ef, "m": M, "qps": nq / ms * 1e3,
                                  "ms_per_batch": ms, "recall@10": rec, "ivf_pq_scan_ms": scan_ms,
                                  "lookups_per_batch": lookups, "lookup_floor_ms": floor_ms,
                                  "scan_over_floor": scan_ms / floor_ms if floor_ms else None,
                                  "rows_visited_per_query": float(visited[:nq].mean()), "oracle_queries": nc,
                                  "gpu_vs_oracle_exact_id_rate": same, **card}), flush=True)
        for ef in (60, 120, 240):
            ms_pq = timed_calls(lambda q, n, i, d, c: L.check(lib.vdb_pq_knn_dev(vs._h, pq._h, p(q), n, k, ef, p(i), p(d), p(c), st)))
            rec_pq = recall_at(ids[:nrec].cpu().numpy(), gt_ids[:nrec])
            print(json.dumps({"config": "Flat knn_pq (same ef)", "nq": nq, "ef": ef, "qps": nq / ms_pq * 1e3, "ms_per_batch": ms_pq,
                              "recall@10": rec_pq, **card}), flush=True)


if __name__ == "__main__":
    main()
