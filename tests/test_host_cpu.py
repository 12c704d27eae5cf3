"""`not gpu`: host logic, the C-ABI library (load + symbols, no compute), and the world_size-2 shard/merge path."""
import ctypes as C
import os
import re
import socket
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    names = set()
    inc = os.path.join(ROOT, "include")
    for fn in os.listdir(inc):
        if fn.endswith(".h"):
            src = open(os.path.join(inc, fn)).read()
            src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
            names |= set(re.findall(r"\b(vdb_[a-z0-9_]+)\s*\(", src))
    return names


def test_library_loads_and_exports_every_declared_symbol():
    import __graft_entry__ as g
    g.build()
    from lab_1806_vec_db_b200 import _lib as L
    lib = C.CDLL(L.LIB_PATH)
    decl = declared_symbols()
    assert len(decl) >= 35
    for name in decl:
        assert hasattr(lib, name), f"{name} is declared in include/ but not exported"
    assert set(L.SIGNATURES) == decl, set(L.SIGNATURES) ^ decl
    assert L.lib().vdb_version() == 801


def test_rust_shim_binds_only_declared_entry_points_with_matching_arity():
    """rust_shim/vdb_b200.rs cannot be compiled here (no Rust toolchain), so its extern block is checked textually:
    every bound function is declared in include/vdb_b200.h with the same number of arguments, and every call site in
    the shim passes that many."""
    hdr = open(os.path.join(ROOT, "include", "vdb_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    shim = open(os.path.join(ROOT, "rust_shim", "vdb_b200.rs")).read()
    shim_nc = re.sub(r"//[^\n]*", "", shim)

    def nargs(arglist):
        arglist = arglist.strip()
        return 0 if arglist in ("", "void") else arglist.count(",") + 1
    c_decl = {m.group(1): nargs(m.group(2)) for m in re.finditer(r"\b(vdb_[a-z0-9_]+)\s*\(([^()]*)\)\s*;", hdr)}
    rs_decl = {m.group(1): nargs(m.group(2)) for m in re.finditer(r"pub fn (vdb_[a-z0-9_]+)\(([^()]*)\)", shim_nc)}
    assert len(rs_decl) >= 30
    for name, n in rs_decl.items():
        assert name in c_decl, f"{name} is bound by the shim but not declared in include/vdb_b200.h"
        assert c_decl[name] == n, f"{name}: header has {c_decl[name]} arguments, shim declares {n}"
    # call sites: `vdb_xxx(` inside `unsafe { ... }` with balanced parentheses
    for m in re.finditer(r"unsafe \{ (vdb_[a-z0-9_]+)\(", shim_nc):
        name, i, depth, commas = m.group(1), m.end(), 1, 0
        empty = True
        while depth:
            ch = shim_nc[i]
            depth += ch in "([{"
            depth -= ch in ")]}"
            commas += ch == "," and depth == 1
            empty &= ch.isspace() or depth == 0
            i += 1
        assert (0 if empty else commas + 1) == rs_decl[name], f"call of {name} passes {commas + 1} arguments"
    assert "gpu_mirror" not in shim  # round-1 finding: the shim called a method that exists nowhere


def test_no_cpu_fallback_on_a_box_without_gpu():
    """The product path must fail loudly, never compute on the CPU."""
    import lab_1806_vec_db_b200 as V
    from conftest import have_gpu
    if have_gpu():
        pytest.skip("a GPU is present")
    with pytest.raises(V.VdbError):
        V.FlatIndex.from_vec_set(np.zeros((4, 8), np.float32), "l2sqr")


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "lab_1806_vec_db_b200")
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".inc", ".h")):
                src = open(os.path.join(dirpath, fn)).read()
                assert "import oracle" not in src and "liboracle" not in src and "orc_" not in src, fn


def test_metric_names_follow_pyo3():
    from lab_1806_vec_db_b200 import _lib as L
    assert L.metric_code("l2sqr") == 0 and L.metric_code("cosine") == 1
    with pytest.raises(ValueError):
        L.metric_code("dot")  # no such DistanceAlgorithm variant (distance/mod.rs:18-28)


def test_key_packing_orders_like_candidate_pair():
    from lab_1806_vec_db_b200.sharded import pack_keys, unpack_keys
    d = np.array([0.0, -0.0, 1.5, -1e-7, np.inf, np.nan, 1.5, 3e-39], np.float32)
    i = np.array([7, 3, 2, 9, 1, 0, 1, 4], np.uint64)
    keys = pack_keys(d, i)
    order = np.argsort(keys, kind="stable")
    # expected: (-1e-7,9) (-0.0,3) (0.0,7) (3e-39,4) (1.5,1) (1.5,2) (inf,1) (nan,0): -0 == +0, NaN greatest
    assert order.tolist() == [3, 1, 0, 7, 6, 2, 4, 5]
    dd, ii = unpack_keys(keys)
    assert (ii == i).all() and np.isnan(dd[5]) and dd[2] == np.float32(1.5) and dd[3] == np.float32(-1e-7)


def test_shard_bounds_cover_everything():
    from lab_1806_vec_db_b200.sharded import shard_bounds
    for n in (0, 1, 7, 1000, 1_000_000):
        for w in (1, 2, 3, 8):
            b = [shard_bounds(n, w, r) for r in range(w)]
            assert b[0][0] == 0 and b[-1][1] == n
            assert all(b[r][1] == b[r + 1][0] for r in range(w - 1))
            assert max(h - l for l, h in b) - min(h - l for l, h in b) <= 1


WORKER = r"""
import os, sys
import numpy as np
import torch, torch.distributed as dist
sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, "tests"))
from lab_1806_vec_db_b200.sharded import shard_bounds, pack_keys, unpack_keys
import oracle as O
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
fx = np.load(os.path.join({root!r}, "tests", "golden", "fixtures.npz"))
dec = lambda u: (u.astype(np.float64) / 1e4).astype(np.float32)
base, test = dec(fx["base_u16"]), dec(fx["test_u16"])[:32]
k = 10
lo, hi = shard_bounds(len(base), world, rank)
ids, dd, cnt = O.flat_knn(base[lo:hi], test, k, "l2sqr")           # this rank's shard (oracle stands in for the GPU)
keys = torch.from_numpy(pack_keys(dd, ids + np.uint64(lo)).astype(np.int64))
allk = [torch.empty_like(keys) for _ in range(world)]
dist.all_gather(allk, keys)                                          # the path's one exchange step
merged = np.sort(np.concatenate([a.numpy().astype(np.uint64) for a in allk], axis=1), axis=1)[:, :k]
md, mi = unpack_keys(merged)
wi, wd, _ = O.flat_knn(base, test, k, "l2sqr")
assert (mi == wi).all() and (md.view(np.uint32) == wd.view(np.uint32)).all()
dist.destroy_process_group()
print("rank", rank, "ok")
"""


def test_world_size_2_shard_and_merge_gloo(tmp_path):
    """Row sharding + all-gather + (distance, id) merge reproduce the unsharded result (CPU, gloo)."""
    script = tmp_path / "worker.py"
    script.write_text(WORKER.format(root=ROOT))
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port), str(script)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert r.stdout.count("ok") == 2


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the GPU arm): one JSON line with the GPU arm's
    metric / unit / config keys, `impl`, `cpu_baseline` and a zero-copy `e2e`; ranks other than 0 print nothing."""
    import json
    import subprocess
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--n", "20000", "--nq", "64",
           "--k", "10", "--steps", "1", "--warmup", "0", "--cpu-queries", "4"]
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "QPS, exact Flat L2 kNN" and d["unit"] == "queries/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["vs_baseline"] is None
    assert d["config"]["n"] == 20000 and d["config"]["nq"] == 64 and d["config"]["k"] == 10 and "workload" in d["config"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    other = subprocess.run(cmd, capture_output=True, text=True, env=dict(env, RANK="1", WORLD_SIZE="2"), timeout=600)
    assert other.returncode == 0 and other.stdout.strip() == ""


def test_bench_dump_outputs_are_the_timed_results_and_repeat(tmp_path):
    """`--dump-outputs DIR`: the last timed step's ids / distances / counts as float .npy files; the same arguments give
    the same inputs, so two runs write the same arrays (here through the CPU arm, checked against the oracle)."""
    import oracle as O
    import bench
    runs = []
    for i in range(2):
        out = tmp_path / f"run{i}"
        cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--n", "20000", "--nq", "64",
               "--k", "10", "--steps", "1", "--warmup", "0", "--cpu-queries", "4", "--dump-outputs", str(out)]
        r = subprocess.run(cmd, capture_output=True, text=True, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        runs.append({n: np.load(out / f"{n}.npy") for n in ("ids", "dist", "counts", "query_rows")})
    a, b = runs
    for n in a:
        assert a[n].dtype in (np.float32, np.float64) and a[n].tobytes() == b[n].tobytes(), n
    assert a["ids"].shape == a["dist"].shape == (4, 10) and a["query_rows"].tolist() == [0, 1, 2, 3]
    base1000, test1000 = bench.load_fixtures()
    base = bench.synth(base1000, 0, 20000, 42, "cpu").numpy()
    q = bench.synth(test1000, 0, 4, 43, "cpu").numpy()
    wi, wd, wc = O.flat_knn(base, q, 10, "l2sqr")
    assert (a["ids"] == wi).all() and (a["dist"] == wd).all() and (a["counts"] == wc).all()
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 2 and "--steps" in r.stderr                      # no run without a timed step


def test_bench_dump_outputs_sample_a_large_batch(tmp_path):
    """Beyond 64 MB in all, a fixed seeded sample of query rows is written, the same one every time."""
    import bench
    nq, k = 70_000, 100
    ids = np.arange(nq * k, dtype=np.int64).reshape(nq, k)
    dist = np.arange(nq * k, dtype=np.float32).reshape(nq, k)
    counts = np.full(nq, k, np.int32)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), ids, dist, counts)
    total = sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a"))
    assert total <= bench.DUMP_BYTES + 4 * 4096                                          # + the .npy headers
    rows = np.load(tmp_path / "a" / "query_rows.npy").astype(np.int64)
    assert 0 < len(rows) < nq and (np.diff(rows) > 0).all()
    assert (np.load(tmp_path / "a" / "ids.npy") == ids[rows]).all()
    assert (np.load(tmp_path / "a" / "dist.npy") == dist[rows]).all()
    for f in os.listdir(tmp_path / "a"):
        assert (tmp_path / "a" / f).read_bytes() == (tmp_path / "b" / f).read_bytes(), f


# ---- rand_compat: the reference's random stream restated (rand 0.8.5 StdRng = ChaCha12) -------------------------------
def test_chacha_core_matches_the_published_keystreams():
    """Zero key, zero nonce, block 0: the keystream vectors published for ChaCha8 / ChaCha12 / ChaCha20 (the eSTREAM /
    IETF test vectors for the original 64-bit-counter layout, which rand_chacha uses). This pins the block function and
    the word order; the seeding and sampling layers above it are restated but cannot be pinned without the crates."""
    from lab_1806_vec_db_b200.rand_compat import chacha_blocks
    want = {
        8: "3e00ef2f895f40d67f5bb8e81f09a5a12c840ec3ce9a7f3b181be188ef711a1e984ce172b9216f419f445367456d5619"
           "314a42a3da86b001387bfdb80e0cfe42",
        12: "9bf49a6a0755f953811fce125f2683d50429c3bb49e074147e0089a52eae155f0564f879d27ae3c02ce82834acfa8c79"
            "3a629f2ca0de6919610be82f411326be",
        20: "76b8e0ada0f13d90405d6ae55386bd28bdd219b8a08ded1aa836efcc8b770dc7da41597c5157488d7724e03fb8d84a37"
            "6a43b8f41518a11cc387b669b2ee6586",
    }
    for rounds, hexes in want.items():
        got = chacha_blocks([0] * 8, 0, 1, rounds).astype("<u4").tobytes().hex()
        assert got == hexes, rounds
    # blocks are consecutive counters: block 1 of a 2-block call = a 1-block call at counter 1
    two = chacha_blocks(list(range(1, 9)), 5, 2, 12)
    assert (two[16:] == chacha_blocks(list(range(1, 9)), 6, 1, 12)).all()
    assert not (two[:16] == two[16:]).all()


def test_stdrng_draws_follow_the_restated_rand_algorithms():
    from lab_1806_vec_db_b200.rand_compat import StdRng, k_means_init_indices
    a, b = StdRng.seed_from_u64(42), StdRng.seed_from_u64(42)
    w = [a.next_u32() for _ in range(6)]
    assert b.next_u64() == w[0] | (w[1] << 32) and b.next_u32() == w[2]        # u64 = two consecutive words, low first
    assert StdRng.seed_from_u64(43).next_u32() != w[0]
    # gen_range: in range, one draw unless rejected, hi word of the widening multiply
    r, s = StdRng.seed_from_u64(7), StdRng.seed_from_u64(7)
    for n in (1, 2, 3, 1000, 10**6, 2**31 + 5, 1 << 20):
        v = r.gen_range_usize(n)
        while True:                                      # accept iff the low half of the product is inside the zone
            x = s.next_u64()
            lo, hi = (x * n) & (2**64 - 1), (x * n) >> 64
            if lo <= ((n << (64 - n.bit_length())) & (2**64 - 1)) - 1:
                break
        assert 0 <= v < n and v == hi
    assert r.next_u32() == s.next_u32()                  # both consumed the same number of words
    draws = [StdRng.seed_from_u64(i).gen_range_u32(10) for i in range(400)]
    assert min(draws) == 0 and max(draws) == 9 and 20 < draws.count(3) < 65
    # shuffle: a permutation, n - 1 draws through the u32 path
    r, s = StdRng.seed_from_u64(1), StdRng.seed_from_u64(1)
    p = r.shuffle(100)
    assert sorted(p.tolist()) == list(range(100)) and p.tolist() != list(range(100))
    for i in range(99, 0, -1):
        s.gen_range_u32(i + 1)
    assert r.next_u32() == s.next_u32()
    # WeightedIndex<f32>: zero weights are never picked, errors are None, the first index above the sample wins
    r = StdRng.seed_from_u64(3)
    picks = [r.weighted_index_f32(np.array([0, 1, 0, 3, 0], np.float32)) for _ in range(300)]
    assert set(picks) == {1, 3} and 40 < picks.count(1) < 120
    assert r.weighted_index_f32(np.zeros(4, np.float32)) is None
    assert r.weighted_index_f32(np.array([1, -1], np.float32)) is None
    assert r.weighted_index_f32(np.array([1, np.nan], np.float32)) is None
    assert StdRng._uniform_f32_scale(0.0, 1.0) == np.float32(1.0)
    u = StdRng.seed_from_u64(9).gen_unit_f32_array(1000)
    assert u.dtype == np.float32 and (u >= 0).all() and (u < 1).all() and ((u * 2.0**23) % 1 == 0).all()
    # k-means++ (k_means.rs:61-87): one usize draw, then per round a weighted sample (one word, skipped when
    # WeightedIndex::new fails) AND the eagerly evaluated fallback draw (always)
    n, k = 50, 5
    r, s = StdRng.seed_from_u64(11), StdRng.seed_from_u64(11)
    got = k_means_init_indices(lambda idx: np.zeros(n, np.float32), n, k, r)
    assert got == [s.gen_range_usize(n) for _ in range(k)]                       # all-zero weights: the fallback wins
    r, s = StdRng.seed_from_u64(12), StdRng.seed_from_u64(12)
    wts = np.linspace(0, 1, n, dtype=np.float32)
    got = k_means_init_indices(lambda idx: wts, n, k, r)
    want = [s.gen_range_usize(n)]
    for _ in range(1, k):
        want.append(s.weighted_index_f32(wts))
        s.gen_range_usize(n)                                                     # drawn and dropped
    assert got == want and r.next_u32() == s.next_u32()
