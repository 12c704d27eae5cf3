"""Flat kNN above the fused top-k: time per call, QPS and the byte model of DESIGN.md section 4 (K1, large k) on the bench
rows (1M x 960 f32, and the same rows as u8), device-resident calls timed with CUDA events. Not the bench.
Usage: python scripts/probe_large_k.py [cases.json]

Per case: ms per call, QPS, modelled bytes and their rate as a fraction of the bandwidth a large device-to-device copy
reaches in the same run, and whether the first k_fused columns equal the fused call at k_fused bit for bit."""
import ctypes as C
import json
import math
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import bench as B  # noqa: E402
import lab_1806_vec_db_b200 as V  # noqa: E402
from lab_1806_vec_db_b200 import _lib as L  # noqa: E402
from test_flat_large_k_gpu import k_fused  # noqa: E402

SEL_ROUNDS, SORT_TILE = 8, 4096
lib = L.lib()
dev = torch.device("cuda:0")
st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
n = int(os.environ.get("N", 1_000_000))
dim = B.DIM


def gpu_facts():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        pl = f"unread ({e})"
    return name, pl


def copy_bandwidth():
    """GB/s of a 4 GiB device-to-device copy (read + write bytes over time)."""
    a = torch.empty(1 << 29, dtype=torch.float64, device=dev)
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 10
    del a, b
    return 2 * (8 << 29) / ms / 1e6


def model_bytes(nq, k, row_bytes):
    """Rows pass per <= 8 queries + per query: 8 N keys written, select (8 rounds + compaction, each reading 8 N; only
    the compaction when k >= N), sort (tile sort read + write, then one read + write per merge pass over kp keys) and
    the decoded results (20 bytes per slot: keys, ids, distances)."""
    rows = math.ceil(nq / 8) * n * row_bytes
    kp = math.ceil(min(k, n) / SORT_TILE) * SORT_TILE
    passes = max(0, math.ceil(math.log2(kp / SORT_TILE))) if kp > SORT_TILE else 0
    reads = (SEL_ROUNDS + 1) if k < n else 1
    per_q = 8 * n + reads * 8 * n + 16 * kp * (1 + passes) + 20 * k
    return rows + nq * per_q


def call(vs, qq, k):
    nq = qq.shape[0]
    ids = torch.empty((nq, k), dtype=torch.int64, device=dev)
    dd = torch.empty((nq, k), dtype=torch.float32, device=dev)
    cnt = torch.empty((nq,), dtype=torch.int32, device=dev)
    f = lambda: L.check(lib.vdb_flat_knn_dev(vs._h, C.c_void_p(qq.data_ptr()), nq, k, C.c_void_p(ids.data_ptr()),  # noqa: E731
                                             C.c_void_p(dd.data_ptr()), C.c_void_p(cnt.data_ptr()), st))
    return f, (ids, dd, cnt)


def timed(f, min_ms=400.0):
    f()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    f()
    e1.record()
    torch.cuda.synchronize()
    reps = max(3, min(200, int(min_ms / max(e0.elapsed_time(e1), 1e-3))))
    e0.record()
    for _ in range(reps):
        f()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, reps


def main():
    name, pl = gpu_facts()
    bw = copy_bandwidth()
    print(f"GPU: {name}, power limit {pl}; 4 GiB device-to-device copy: {bw:.0f} GB/s", flush=True)
    b1000, t1000 = B.load_fixtures()
    base = B.synth(b1000, 0, n, 42, dev)
    qf = B.synth(t1000, 0, 100, 43, dev)
    out = {"gpu": name, "power_limit": pl, "copy_gbs": bw, "n": n, "dim": dim, "cases": []}
    for dtype in ("f32", "u8"):
        rows = base if dtype == "f32" else (base * 255).round().to(torch.uint8)
        qs = qf if dtype == "f32" else (qf * 255).round().to(torch.uint8)
        npdt = np.float32 if dtype == "f32" else np.uint8
        vs = V.DeviceVecSet.from_device(rows.data_ptr(), n, dim, dim, npdt, "l2sqr", keepalive=rows)
        row_bytes = dim * (4 if dtype == "f32" else 1)
        for nq in (1, 8, 100):
            qq = qs[:nq].contiguous()
            kf = k_fused(dim, npdt, nq)
            f, ref = call(vs, qq, kf)
            f()
            torch.cuda.synchronize()
            ref_ids, ref_d = ref[0].cpu().numpy(), ref[1].cpu().numpy()
            ks = ([10] if nq == 1 else []) + [kf, kf + 1, 100_000, 1_000_000]
            for k in ks:
                f, res = call(vs, qq, k)
                ms, reps = timed(f)
                same = None
                if k >= kf:
                    c = min(k, kf)
                    same = bool((res[0][:, :c].cpu().numpy() == ref_ids[:, :c]).all() and
                                (res[1][:, :c].cpu().numpy().view(np.uint32) == ref_d[:, :c].view(np.uint32)).all())
                mb = model_bytes(nq, k, row_bytes) if k > kf else None
                case = {"dtype": dtype, "nq": nq, "k": k, "k_fused": kf, "ms": round(ms, 4), "reps": reps,
                        "qps": round(nq / ms * 1e3, 1), "prefix_bit_identical": same}
                line = f"{dtype} nq={nq:3d} k={k:8d} (k_fused {kf}): {ms:9.3f} ms/call  {nq / ms * 1e3:9.1f} QPS"
                if mb is not None:
                    case["model_bytes"] = mb
                    case["model_frac_of_copy_bw"] = round(mb / ms / 1e6 / bw, 3)
                    line += f"  model {mb / 1e9:7.2f} GB -> {case['model_frac_of_copy_bw'] * 100:5.1f}% of copy bandwidth"
                if same is not None:
                    line += f"  first {min(k, kf)} columns bit-identical to k_fused: {same}"
                print(line, flush=True)
                out["cases"].append(case)
                del res, f
                torch.cuda.empty_cache()
        del vs, rows
    print(f"GPU: {name}, power limit {pl}", flush=True)
    if len(sys.argv) > 1:   # optional: the cases as JSON
        with open(sys.argv[1], "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
