"""One workload family of the switch matrix (tests/switch_matrix.py), run in a process of its own.

    python tests/switch_child.py <family> <out.npz>

Builds the family's seeded inputs, runs its calls under torch.profiler (CUDA activities) and writes every output array
(ids, distances, counts; codes and graph links where the family has them) plus `__fingerprint__`: one line
"kernel name | grid | block | shared memory" per kernel launch of the calls (a multiset: the parent compares counts).
The shared memory of a trace event is static + dynamic; the static part is fixed per kernel, so two launches of one
kernel differ there only by their dynamic shared memory. A trace without kernel events is an error (exit code 3).

Most switches are read once per process, so each (switch, value) needs a fresh process; the input builders are also
imported by tests/test_switches_gpu.py to check the default run against the CPU oracle.
"""
import json
import os
import sys
import tempfile
from collections import Counter

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

KEY_NONE = np.uint64(0xFFFFFFFFFFFFFFFF)


def clustered(n, nq, dim, seed, nproto=256, dtype=np.float32):
    """Rows and queries around shared prototypes (as tests/test_multi_gpu.py::_data): thresholds and pruning bounds
    decide something, unlike on a uniform cloud."""
    rng = np.random.default_rng(seed)
    proto = rng.random((nproto, dim), dtype=np.float32) * 0.15
    base = (proto[rng.integers(0, nproto, n)] + 0.02 * rng.standard_normal((n, dim), dtype=np.float32)).clip(0, 1)
    q = (proto[rng.integers(0, nproto, nq)] + 0.02 * rng.standard_normal((nq, dim), dtype=np.float32)).clip(0, 1)
    if dtype == np.uint8:
        return (base * 255).astype(np.uint8), (q * 255).astype(np.uint8)
    return base.astype(np.float32), q.astype(np.float32)


# ---- Flat tensor path ---------------------------------------------------------------------------------------------
# f32: 782 row tiles of 256; nq = 64 on single CTAs has a slab cap of 6 tiles (VDB_GEMM_TPS=8 shrinks the grid),
#      nq = 300 runs on CTA pairs, nq = 5000 is long enough for the chunk pipeline, k = 300 takes the two-level sample.
# u8s: 274 row tiles: nq = 64 has a slab cap of 2 (VDB_GEMM_TPS=1 widens the grid).
# u8l: a 32768-row sample (128 tiles): nq = 5000 puts 17 tiles in a sample slab by default, so VDB_GEMM_SAMPLE_TPS=32
#      and =1 change the number of slabs the sample merge reads.
FLAT_SETS = {"f32": (200_000, 100, np.float32, 1), "u8s": (70_000, 100, np.uint8, 2), "u8l": (1_000_000, 32, np.uint8, 3)}
FLAT_CALLS = [  # (set, metric, nq, k, force_redo)
    ("f32", "l2sqr", 300, 10, 0), ("f32", "l2sqr", 300, 300, 0), ("f32", "l2sqr", 64, 10, 0),
    ("f32", "l2sqr", 5000, 10, 0), ("f32", "l2sqr", 5000, 10, 3),
    ("f32", "cosine", 300, 10, 0), ("f32", "cosine", 300, 300, 0), ("f32", "cosine", 64, 10, 0),
    ("u8s", "l2sqr", 64, 10, 0), ("u8s", "l2sqr", 300, 10, 0),
    ("u8l", "l2sqr", 5000, 10, 0),
]


def flat_inputs():
    out = {}
    for name, (n, dim, dtype, seed) in FLAT_SETS.items():
        base, q = clustered(n, 5000, dim, seed, dtype=dtype)
        base[n // 2] = base[123]            # an exact duplicate: the lower id comes first
        q[0] = base[123]
        out[name] = (base, q)
    return out


def flat_key(s, metric, nq, k, redo):
    return f"flat/{s}/{metric}/nq{nq}/k{k}" + (f"/redo{redo}" if redo else "")


def run_flat():
    import lab_1806_vec_db_b200 as V
    from lab_1806_vec_db_b200 import _lib as L
    lib = L.lib()
    sets = flat_inputs()
    res = {}
    L.check(lib.vdb_flat_set_path(2))     # the tensor route for every batch size
    try:
        for s, metric in dict.fromkeys((c[0], c[1]) for c in FLAT_CALLS):
            base, q = sets[s]
            idx = V.FlatIndex.from_vec_set(base, metric)
            for s2, m2, nq, k, redo in FLAT_CALLS:
                if (s2, m2) != (s, metric):
                    continue
                L.check(lib.vdb_debug_force_redo(redo))
                key = flat_key(s, metric, nq, k, redo)
                res[key + "/ids"], res[key + "/dist"], res[key + "/counts"] = idx.knn_batch(q[:nq], k)
                L.check(lib.vdb_debug_force_redo(0))
            idx.vec_set.close()
    finally:
        L.check(lib.vdb_debug_force_redo(0))
        L.check(lib.vdb_flat_set_path(0))
    return res


# ---- key merges: the C ABI merges and a row-sharded Flat search on devices [0, 0, 0] -----------------------------
MERGE_SHAPES = ((8, 37, 100), (2, 5, 10), (5, 3, 600), (3, 4, 1), (4, 300, 64))   # (nlists, nq, k)
MERGE_SHARDED_CALLS = (("l2sqr", 300, 10), ("l2sqr", 300, 100), ("l2sqr", 5, 10), ("cosine", 300, 10))


def merge_lists(nlists, nq, k, seed):
    """Ascending per-list keys with KEY_NONE padding, short lists and keys shared between lists."""
    rng = np.random.default_rng(seed)
    lists = np.full((nlists, nq, k), KEY_NONE, np.uint64)
    for li in range(nlists):
        for q in range(nq):
            cnt = int(rng.integers(0, k + 1))
            vals = rng.integers(0, 1 << 40, cnt).astype(np.uint64)
            if li and cnt and rng.random() < 0.5:      # a key that also occurs in list 0
                src = lists[0, q][lists[0, q] != KEY_NONE]
                if len(src):
                    vals[0] = src[0]
            lists[li, q, :cnt] = np.sort(vals)
    return lists


def merge_sharded_inputs():
    base, q = clustered(150_000, 300, 64, 4)
    base[100_000] = base[123]           # a duplicate in another shard
    return base, q


def run_merge():
    import ctypes as C
    import torch
    import lab_1806_vec_db_b200 as V
    from lab_1806_vec_db_b200 import _lib as L
    lib = L.lib()
    res = {}
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for i, (nlists, nq, k) in enumerate(MERGE_SHAPES):
        d = torch.from_numpy(merge_lists(nlists, nq, k, 8 + i).view(np.int64)).cuda()
        out = torch.empty((nq, k), dtype=torch.int64, device="cuda")
        L.check(lib.vdb_merge_keys_to_keys_dev(C.c_void_p(d.data_ptr()), nlists, nq, k, C.c_void_p(out.data_ptr()), st))
        ids = torch.empty((nq, k), dtype=torch.int64, device="cuda")
        dd = torch.empty((nq, k), dtype=torch.float32, device="cuda")
        cnt = torch.empty((nq,), dtype=torch.int32, device="cuda")
        L.check(lib.vdb_merge_keys_dev(C.c_void_p(d.data_ptr()), nlists, nq, k, C.c_void_p(ids.data_ptr()),
                                       C.c_void_p(dd.data_ptr()), C.c_void_p(cnt.data_ptr()), st))
        torch.cuda.synchronize()
        key = f"merge/{nlists}x{nq}x{k}"
        res[key + "/keys"] = out.cpu().numpy().view(np.uint64)
        res[key + "/ids"] = ids.cpu().numpy().view(np.uint64)
        res[key + "/dist"] = dd.cpu().numpy()
        res[key + "/counts"] = cnt.cpu().numpy()
    base, q = merge_sharded_inputs()
    V.init_devices([0, 0, 0])
    try:
        for metric in dict.fromkeys(c[0] for c in MERGE_SHARDED_CALLS):
            idx = V.FlatIndex.from_vec_set(base, metric)
            assert len(idx.vec_set.shards()) == 3
            for m2, nq, k in MERGE_SHARDED_CALLS:
                if m2 == metric:
                    key = f"sharded/{metric}/nq{nq}/k{k}"
                    res[key + "/ids"], res[key + "/dist"], res[key + "/counts"] = idx.knn_batch(q[:nq], k)
            idx.vec_set.close()
    finally:
        V.init_devices([])
    return res


# ---- IVF probe scan -----------------------------------------------------------------------------------------------
IVF_N, IVF_DIM, IVF_NLIST = 100_000, 64, 64
IVF_CALLS = [  # (metric, nq, k, nprobe): 600 queries put > 128 queries on some lists (CTA-pair tiles)
    ("l2sqr", 600, 10, 4), ("l2sqr", 600, 100, 2), ("l2sqr", 40, 10, 4),
    ("cosine", 600, 10, 4), ("cosine", 40, 100, 3),
]


def ivf_inputs():
    rng = np.random.default_rng(5)
    proto = rng.random((IVF_NLIST, IVF_DIM), dtype=np.float32)
    base = (proto[rng.integers(0, IVF_NLIST, IVF_N)] + 0.08 * rng.standard_normal((IVF_N, IVF_DIM))).astype(np.float32)
    base[3000:3040] = base[11]          # ties decided by id
    owner = np.concatenate([np.repeat(np.arange(3), 160), rng.integers(0, IVF_NLIST, 120)])   # 160 queries on lists 0-2
    q = (proto[owner] + 0.08 * rng.standard_normal((len(owner), IVF_DIM))).astype(np.float32)
    q[1] = base[11]
    return base, proto, q


def run_ivf():
    import lab_1806_vec_db_b200 as V
    base, cent, q = ivf_inputs()
    res = {}
    for metric in dict.fromkeys(c[0] for c in IVF_CALLS):
        vs = V.DeviceVecSet(base, metric)
        ivf = V.IVFIndex(vs, cent)
        res[f"ivf/{metric}/assignment"] = np.asarray(ivf.assignment)
        for m2, nq, k, nprobe in IVF_CALLS:
            if m2 == metric:
                key = f"ivf/{metric}/nq{nq}/k{k}/p{nprobe}"
                res[key + "/ids"], res[key + "/dist"], res[key + "/counts"] = ivf.knn_with_ef_batch(q[:nq], k, nprobe)
        ivf.close()
        vs.close()
    return res


# ---- PQ: encode and every ADC scan ----------------------------------------------------------------------------------
PQ_N, PQ_DIM = 70_000, 64
PQ_TABLES = [  # (name, dtype, metric, m, n_bits)
    ("f32_l2_m32", np.float32, "l2sqr", 32, 4),      # 2-dim sub-vectors: one-hot contraction
    ("f32_l2_m16", np.float32, "l2sqr", 16, 4),      # 4-dim sub-vectors: decoded contraction
    ("f32_cos_m32", np.float32, "cosine", 32, 4),    # cosine: no tensor filter
    ("f32_l2_m16_b8", np.float32, "l2sqr", 16, 8),   # 8-bit: per-CTA scan only
    ("u8_l2_m32", np.uint8, "l2sqr", 32, 4),
    ("u8_cos_m16", np.uint8, "cosine", 16, 4),
]
PQ_CALLS = [(1, 10, 50), (2, 10, 50), (3, 10, 50), (8, 10, 50), (8, 5, 300), (64, 10, 50), (64, 5, 300)]   # (nq, k, ef)


def pq_inputs():
    sets = {}
    for dtype, seed in ((np.float32, 6), (np.uint8, 7)):
        base, q = clustered(PQ_N, 64, PQ_DIM, seed, dtype=dtype)
        base[5000:5300] = base[17]      # 300 identical rows: ADC ties decided by id
        q[0] = base[17]
        sets[np.dtype(dtype).name] = (base, q)
    return sets


def pq_books(V, base, m, n_bits):
    kc = 1 << n_bits
    return np.concatenate([np.ascontiguousarray(base[100:100 + kc, lo:hi]).reshape(-1) for lo, hi in V.pq_groups(base.shape[1], m)])


def run_pq():
    import lab_1806_vec_db_b200 as V
    sets = pq_inputs()
    res = {}
    for name, dtype, metric, m, n_bits in PQ_TABLES:
        base, q = sets[np.dtype(dtype).name]
        vs = V.DeviceVecSet(base, metric)
        pq = V.PQTable(vs, V.PQConfig(n_bits, m, metric), pq_books(V, base, m, n_bits))
        res[f"pq/{name}/codes"] = pq.encoded_vec_set.copy()
        idx = V.FlatIndex(vs)
        for nq, k, ef in PQ_CALLS:
            key = f"pq/{name}/nq{nq}/k{k}/ef{ef}"
            res[key + "/ids"], res[key + "/dist"], res[key + "/counts"] = idx.knn_pq_batch(q[:nq], k, ef, pq)
        pq.close()
        vs.close()
    return res


# ---- HNSW ---------------------------------------------------------------------------------------------------------
HNSW_N, HNSW_DIM, HNSW_M, HNSW_EFC = 20_000, 48, 16, 200
HNSW_EFS = (64, 300)   # 300: the 8192-slot visited set by default, 16384 slots under VDB_HNSW_SMALL_HASH_EF=0 / 200


def hnsw_inputs():
    import lab_1806_vec_db_b200 as V
    base, q = clustered(HNSW_N, 200, HNSW_DIM, 9, nproto=200)
    levels = V.hnsw_rand_levels(HNSW_N, HNSW_M, np.random.default_rng(5))
    return base, q, levels


def run_hnsw():
    import lab_1806_vec_db_b200 as V
    base, q, levels = hnsw_inputs()
    res = {}
    vs = V.DeviceVecSet(base, "l2sqr")
    idx = V.HNSWIndex(vs, V.HNSWConfig(0, HNSW_EFC, HNSW_M), levels=levels)
    res["hnsw/links0"], res["hnsw/len0"] = idx.level0_links()
    res["hnsw/levels"], res["hnsw/ulinks"], res["hnsw/ulen"] = idx.upper_links()
    res["hnsw/enter_point"] = np.array(idx.enter_point, np.int64)
    for ef in HNSW_EFS:
        key = f"hnsw/ef{ef}"
        res[key + "/ids"], res[key + "/dist"], res[key + "/counts"] = idx.knn_with_ef_batch(q, 10, ef)
    return res


RUNS = {"flat": run_flat, "merge": run_merge, "ivf": run_ivf, "pq": run_pq, "hnsw": run_hnsw}


def fingerprint(fn):
    """Runs fn() under torch.profiler (CUDA activities) -> (fn's result, Counter of kernel launch configurations).
    Raises when the trace holds no kernel event: a missing fingerprint must never pass as an unchanged route."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.zeros(1, device="cuda")       # context and the profiler's CUDA side up before the window opens
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    fd, path = tempfile.mkstemp(suffix=".json")
    os.close(fd)
    try:
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    finally:
        os.unlink(path)
    fp = Counter()
    for e in events:
        if e.get("cat") != "kernel":
            continue
        a = e.get("args", {})
        fp[f"{e['name']} | grid {tuple(a.get('grid', ()))} | block {tuple(a.get('block', ()))} | "
           f"smem {a.get('shared memory')}"] += 1
    if not fp:
        raise RuntimeError("the profiler trace holds no kernel events")
    return out, fp


def main(argv):
    if len(argv) != 3 or argv[1] not in RUNS:
        print(f"usage: {argv[0]} <{'|'.join(RUNS)}> <out.npz>", file=sys.stderr)
        return 2
    try:
        res, fp = fingerprint(RUNS[argv[1]])
    except RuntimeError as e:
        if "no kernel events" not in str(e):
            raise
        print(e, file=sys.stderr)
        return 3
    lines = np.array([k for k, c in sorted(fp.items()) for _ in range(c)])
    np.savez(argv[2], __fingerprint__=lines, **{k: np.asarray(v) for k, v in res.items()})
    return 0


if __name__ == "__main__":
    sys.exit(main(sys.argv))
