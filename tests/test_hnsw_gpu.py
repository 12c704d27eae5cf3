"""HNSW on the device (hnsw.cu) vs the single-thread CPU restatement of hnsw_index.rs (oracle) and exact Flat results.
The reference's graph is RNG / thread-count dependent, so parity is: identical algorithm on identical levels
(sequential insertion reproduces the oracle's adjacency almost everywhere), recall@10 not below the oracle's, the
reference's own unit test (ids == Flat ids), structural invariants, and cached-form distances within the parity tolerance."""
import numpy as np
import pytest

from conftest import RTOL, close

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def V():
    import lab_1806_vec_db_b200 as V
    return V


def recall(ids, gt):
    return float(np.mean([len(set(a.tolist()) & set(b.tolist())) / len(b) for a, b in zip(ids, gt)]))


def check_graph(links, lens, n, M):
    assert lens.max() <= 2 * M
    for i in range(n):
        row = links[i, :lens[i]]
        assert (row < n).all() and (row != i).all(), f"bad link at node {i}"
        assert len(set(row.tolist())) == len(row), f"duplicate link at node {i}"
    assert (lens[1:] > 0).all() or n < 3


@pytest.mark.parametrize("metric", ["l2sqr", "cosine"])
def test_hnsw_gist_1000_vs_oracle(V, fixtures, oracle, metric):
    from oracle.oracle_py import HnswOracle
    base, test = fixtures["base"], fixtures["test"][:200]
    M, efc = 16, 200
    levels = V.hnsw_rand_levels(len(base), M, np.random.default_rng(5))
    ref = HnswOracle(base, metric, M, efc, levels)
    vs = V.DeviceVecSet(base, metric)
    idx = V.HNSWIndex(vs, V.HNSWConfig(0, efc, M), levels=levels)
    assert idx.default_ef == 100 and idx.ef_construction == 200
    ep = idx.enter_point
    top = int(levels.max())
    assert ep == (int(np.argmax(levels == top)), top)   # first row that reaches the highest level
    links, lens = idx.level0_links()
    check_graph(links, lens, len(base), M)
    gt = oracle.flat_knn(base, test, 10, metric, nthreads=8)[0]
    row_cache = np.array([oracle.dist_cache(v, metric) for v in base], np.float32)
    for ef in (10, 50, 100):
        ids, dd, cnt = idx.knn_with_ef_batch(test, 10, ef)
        oi, od, oc = ref.knn(test, 10, ef, nthreads=8)
        r_gpu, r_cpu = recall(ids, gt), recall(oi, gt)
        assert r_gpu >= r_cpu - 0.02, (ef, r_gpu, r_cpu)
        assert (cnt == 10).all()
        assert (np.diff(dd, axis=1) >= 0).all()
        # returned distances are the reference's cached form (distance/mod.rs:54-57, 67-69)
        for qi in (0, 7, 199):
            qc = oracle.dist_cache(test[qi], metric)
            want = oracle.gather_dist(base, row_cache, test[qi], qc, ids[qi], metric)
            assert close(dd[qi], want, RTOL, 2e-6).all()
    assert recall(idx.knn_with_ef_batch(test, 10, 100)[0], gt) >= 0.99
    # single-query trait call == batch row
    one = idx.knn_with_ef(test[3], 10, 50)
    many = idx.knn_with_ef_batch(test, 10, 50)
    assert [p.index for p in one] == many[0][3].tolist()


def test_hnsw_sequential_insertion_reproduces_the_oracle_graph(V, fixtures, oracle):
    """max_batch = 1 is the reference's `add` path: same candidates, same heuristic, same back-link pruning. Only
    the summation order of the dot products differs from the CPU, so almost every adjacency list must be identical."""
    from oracle.oracle_py import HnswOracle
    base = fixtures["base"][:600]
    M, efc = 8, 40
    levels = V.hnsw_rand_levels(len(base), M, np.random.default_rng(11))
    ref_links, ref_lens = HnswOracle(base, "l2sqr", M, efc, levels).links0()
    vs = V.DeviceVecSet(base, "l2sqr")
    old = V.HNSWIndex.MAX_BATCH
    V.HNSWIndex.MAX_BATCH = 1
    try:
        idx = V.HNSWIndex(vs, V.HNSWConfig(0, efc, M), levels=levels)
    finally:
        V.HNSWIndex.MAX_BATCH = old
    links, lens = idx.level0_links()
    check_graph(links, lens, len(base), M)
    same = sum(1 for i in range(len(base))
               if lens[i] == ref_lens[i] and set(links[i, :lens[i]].tolist()) == set(ref_links[i, :ref_lens[i]].tolist()))
    assert same >= 0.95 * len(base), same


def test_hnsw_reference_unit_test_shape(V, fixtures, oracle):
    """hnsw_index.rs:776-786: dim clipped to 12, k = 6, query = row 200: the ids equal the Flat index's ids."""
    base = np.ascontiguousarray(fixtures["base"][:, :12])
    vs = V.DeviceVecSet(base, "l2sqr")
    idx = V.HNSWIndex(vs, V.HNSWConfig(0, 200, 16), rng=np.random.default_rng(42))
    got = idx.knn(base[200], 6)
    want = oracle.flat_knn(base, base[200:201], 6, "l2sqr")[0][0]
    assert [p.index for p in got] == want.tolist()
    assert got[0].index == 200 and abs(got[0].distance) < 1e-6
    with pytest.raises(ValueError):
        idx.knn_with_ef(base[0], 3, 0)
    with pytest.raises(ValueError):
        idx.knn_with_ef(base[0, :5], 3, 10)


def test_hnsw_batched_build_20k_and_u8(V, oracle):
    """Batches of up to 2048 new nodes (read-only search + in-batch brute force + grouped back-links): recall must match
    the sequentially built CPU graph; also u8 rows, k > ef, ef larger than the set."""
    from oracle.oracle_py import HnswOracle
    rng = np.random.default_rng(3)
    n, dim, M, efc = 20_000, 64, 12, 100
    proto = rng.random((200, dim), dtype=np.float32)
    base = (proto[rng.integers(0, 200, n)] + 0.1 * rng.standard_normal((n, dim))).astype(np.float32)
    q = (proto[rng.integers(0, 200, 300)] + 0.1 * rng.standard_normal((300, dim))).astype(np.float32)
    levels = V.hnsw_rand_levels(n, M, rng)
    ref = HnswOracle(base, "l2sqr", M, efc, levels)
    vs = V.DeviceVecSet(base, "l2sqr")
    idx = V.HNSWIndex(vs, V.HNSWConfig(0, efc, M), levels=levels)
    links, lens = idx.level0_links()
    check_graph(links, lens, n, M)
    gt = oracle.flat_knn(base, q, 10, "l2sqr", nthreads=8)[0]
    for ef in (20, 60, 200):
        r_gpu = recall(idx.knn_with_ef_batch(q, 10, ef)[0], gt)
        r_cpu = recall(ref.knn(q, 10, ef, nthreads=8)[0], gt)
        assert r_gpu >= r_cpu - 0.03, (ef, r_gpu, r_cpu)
    ids, dd, cnt = idx.knn_with_ef_batch(q[:4], 30, 5)    # ef = max(ef, k)
    assert (cnt == 30).all()
    # u8 rows
    b8 = rng.integers(0, 256, (3000, 48)).astype(np.uint8)
    q8 = b8[:50].copy()
    vs8 = V.DeviceVecSet(b8, "l2sqr")
    i8 = V.HNSWIndex(vs8, V.HNSWConfig(0, 64, 8), rng=rng)
    ids, dd, cnt = i8.knn_with_ef_batch(q8, 1, 64)
    assert (ids[:, 0] == np.arange(50)).mean() >= 0.98 and (dd[ids[:, 0] == np.arange(50), 0] == 0).all()
    # tiny sets
    t = V.HNSWIndex(V.DeviceVecSet(base[:3], "l2sqr"), V.HNSWConfig(0, 10, 4), rng=rng)
    ids, dd, cnt = t.knn_with_ef_batch(base[:2], 5, 10)
    assert (cnt == 3).all() and ids[0, 0] == 0 and ids[1, 0] == 1


@pytest.mark.parametrize("metric", ["l2sqr", "cosine"])
def test_hnsw_knn_pq_vs_oracle(V, fixtures, oracle, metric):
    """HNSWIndex::knn_pq (hnsw_index.rs:672-697): graph walk with ADC distances + exact resort of all ef results. Same
    levels, codebooks and codes on both sides; the graphs are built independently, so compare by recall and check the
    returned distances against the cached form."""
    from oracle.oracle_py import HnswOracle
    base, test = fixtures["base"], fixtures["test"][:150]
    M, efc, m = 16, 200, 96
    rng = np.random.default_rng(9)
    levels = V.hnsw_rand_levels(len(base), M, rng)
    books = np.concatenate([np.ascontiguousarray(base[100:116, lo:hi]).reshape(-1) for lo, hi in V.pq_groups(960, m)])
    vs = V.DeviceVecSet(base, metric)
    pq = V.PQTable(vs, V.PQConfig(4, m, metric), books)
    codes = oracle.pq_encode(base, books, m, 4, metric, nthreads=8)
    assert (pq.encoded_vec_set == codes).all()
    idx = V.HNSWIndex(vs, V.HNSWConfig(0, efc, M), levels=levels)
    ref = HnswOracle(base, metric, M, efc, levels)
    gt = oracle.flat_knn(base, test, 10, metric, nthreads=8)[0]
    row_cache = np.array([oracle.dist_cache(v, metric) for v in base], np.float32)
    for ef in (20, 100):
        ids, dd, cnt = idx.knn_pq_batch(test, 10, ef, pq)
        oi, od, oc = ref.knn_pq(test, 10, ef, codes, books, m, 4, nthreads=8)
        r_gpu, r_cpu = recall(ids, gt), recall(oi, gt)
        assert r_gpu >= r_cpu - 0.03, (ef, r_gpu, r_cpu)
        assert (cnt == 10).all() and (np.diff(dd, axis=1) >= 0).all()
        for qi in (0, 5):
            want = oracle.gather_dist(base, row_cache, test[qi], oracle.dist_cache(test[qi], metric), ids[qi], metric)
            assert close(dd[qi], want, RTOL, 2e-6).all()
    one = idx.knn_pq(test[2], 10, 100, pq)
    assert [p.index for p in one] == idx.knn_pq_batch(test, 10, 100, pq)[0][2].tolist()


def test_hnsw_bincode_round_trip_and_oracle_graph_import(V, fixtures, oracle):
    """The device graph is written in the reference's bincode HNSWIndex layout (save_without_vec_set, :642-655), read
    back and re-created over the same rows (load_with_external_vec_set, :656-668): identical search results. A graph
    built by the CPU restatement is imported the same way and searched on the device: ids equal the CPU search."""
    from lab_1806_vec_db_b200 import formats as F
    from oracle.oracle_py import HnswOracle
    base, test = fixtures["base"][:700], fixtures["test"][:64]
    M, efc = 8, 60
    levels = V.hnsw_rand_levels(len(base), M, np.random.default_rng(21))
    vs = V.DeviceVecSet(base, "l2sqr")
    idx = V.HNSWIndex(vs, V.HNSWConfig(len(base), efc, M), levels=levels)
    rec = F.hnsw_index_record(idx)
    blob = F.dump_hnsw_index(rec)
    back = F.load_hnsw_index(blob)
    assert back.m == M and back.max_m0 == 2 * M and back.ef_construction == efc and back.vec_set.shape == (0, 960)
    assert (back.vec_level == levels).all() and [len(o) for o in back.other_links] == (levels * M).tolist()
    idx2 = V.HNSWIndex.from_record(vs, back)
    a, b = idx.knn_with_ef_batch(test, 10, 50), idx2.knn_with_ef_batch(test, 10, 50)
    assert (a[0] == b[0]).all() and (a[1].view(np.uint32) == b[1].view(np.uint32)).all()
    # CPU-built graph -> record -> device
    ref = HnswOracle(base, "l2sqr", M, efc, levels)
    l0, n0 = ref.links0()
    ul, un = ref.upper()
    lens, other, o = [], [], 0
    for i, lv in enumerate(levels):
        lv = int(lv)
        other.append(ul[o * M:(o + lv) * M])
        lens.append(np.concatenate([[n0[i]], un[o:o + lv]]).astype(np.uint64))
        o += lv
    top = int(levels.max())
    rec2 = back._replace(level0_links=l0.reshape(-1), other_links=other, links_len=lens,
                         enter_level=top, enter_point=int(np.argmax(levels == top)))
    idx3 = V.HNSWIndex.from_record(vs, F.load_hnsw_index(F.dump_hnsw_index(rec2)))
    got = idx3.knn_with_ef_batch(test, 10, 50)[0]
    want = ref.knn(test, 10, 50, nthreads=8)[0]
    assert (got == want).mean() >= 0.995       # same graph, same algorithm; only fp summation order differs
    with pytest.raises(V.VdbError):
        V.HNSWIndex.from_record(vs, rec2._replace(level0_links=np.full_like(rec2.level0_links, 5000)))


def test_hnsw_incremental_add_matches_one_shot_build(V, fixtures, oracle):
    """IndexBuilder::batch_add on a built index: rows pushed after the build are inserted into the existing graph.
    With the same levels the result is the graph of a one-shot build whose batches end at the same row (same batch
    pipeline), so build(600) + add(400) with max_batch 1 equals build(1000) with max_batch 1; recall stays at the
    one-shot level for batched adds."""
    base, test = fixtures["base"], fixtures["test"][:100]
    M, efc = 8, 60
    levels = V.hnsw_rand_levels(1000, M, np.random.default_rng(4))
    old = V.HNSWIndex.MAX_BATCH
    try:
        V.HNSWIndex.MAX_BATCH = 1
        one = V.HNSWIndex(V.DeviceVecSet(base, "l2sqr"), V.HNSWConfig(0, efc, M), levels=levels)
        vs = V.DeviceVecSet(base[:600], "l2sqr")
        inc = V.HNSWIndex(vs, V.HNSWConfig(0, efc, M), levels=levels[:600])
        vs.push(base[600:])
        inc.batch_add_pushed(levels=levels[600:])
    finally:
        V.HNSWIndex.MAX_BATCH = old
    a, b = one.level0_links(), inc.level0_links()
    assert (a[1] == b[1]).all() and (a[0] == b[0]).all()
    assert one.enter_point == inc.enter_point
    la, lb = one.upper_links(), inc.upper_links()
    assert all((x == y).all() for x, y in zip(la, lb))
    # batched add (default batch size), searched
    vs2 = V.DeviceVecSet(base[:300], "l2sqr")
    idx = V.HNSWIndex(vs2, V.HNSWConfig(0, 200, 16), rng=np.random.default_rng(1))
    for lo in (300, 301, 650):
        hi = {300: 301, 301: 650, 650: 1000}[lo]
        vs2.push(base[lo:hi])
        idx.batch_add_pushed(np.random.default_rng(lo))
    assert len(idx) == 1000
    gt = oracle.flat_knn(base, test, 10, "l2sqr", nthreads=8)[0]
    assert recall(idx.knn_with_ef_batch(test, 10, 100)[0], gt) >= 0.99
    links, lens = idx.level0_links()
    check_graph(links, lens, 1000, 16)


def test_large_ef_uses_the_global_visited_set_and_matches_the_oracle_on_the_same_graph(V, oracle):
    """ef >= 2048: at ~10 fresh nodes per expansion a shared-memory visited set (28 672 usable slots) would fill up and
    silently drop neighbours; the set now lives in global memory for ef > 896. Parity is checked the strong way: the
    oracle's knn_with_ef walks the VERY graph the GPU built (orc_hnsw_from_graph), so both searches must return the same
    ids (up to near-ties of the cached-form distance), and no search may have overflowed."""
    import ctypes as C
    from oracle.oracle_py import HnswOracle
    rng = np.random.default_rng(21)
    n, dim, M = 30_000, 48, 16
    base = rng.random((n, dim), dtype=np.float32)
    q = rng.random((40, dim), dtype=np.float32)
    vs = V.DeviceVecSet(base, "l2sqr")
    idx = V.HNSWIndex(vs, V.HNSWConfig(0, 200, M), rng=np.random.default_rng(3))
    links0, len0 = idx.level0_links()
    levels, ulinks, ulen = idx.upper_links()
    ep, el = idx.enter_point
    cpu = HnswOracle.from_graph(base, "l2sqr", M, 200, levels, links0, len0, ulinks, ulen, ep, el)
    gt = V.FlatIndex(vs).knn_batch(q, 10)[0]
    for ef in (64, 2048, 4096):
        ids, dd, cnt = idx.knn_with_ef_batch(q, 10, ef)
        oi, od, _ = cpu.knn(q, 10, ef, nthreads=8)
        same = (ids.astype(np.int64) == oi.astype(np.int64))
        assert same.mean() >= 0.98, (ef, float(same.mean()))
        assert np.allclose(dd, od, rtol=1e-4, atol=1e-5)
        if ef >= 2048:
            assert recall(ids, gt) >= 0.999      # ef far above k on 30k rows: the walk reaches every true neighbour
    ov = C.c_uint32(7)
    V._lib.check(V.lib().vdb_hnsw_overflow(idx._h, C.byref(ov)))
    assert ov.value == 0


def test_a_full_visited_set_is_searched_again_not_a_silent_loss(V, tmp_path):
    """With the visited set forced down to 64 slots every search overflows it: the build's batches and the host searches
    run again with a set that cannot fill, so the graph and the results are the default run's bits."""
    import subprocess, sys, textwrap, os
    # the override is read once per process: both runs in children
    code = textwrap.dedent("""
        import numpy as np, sys
        sys.path.insert(0, %r)
        import lab_1806_vec_db_b200 as V
        rng = np.random.default_rng(22)
        base = rng.random((5000, 32), dtype=np.float32)
        idx = V.HNSWIndex(V.DeviceVecSet(base, "l2sqr"), V.HNSWConfig(0, 40, 8), rng=np.random.default_rng(1))
        ids, dd, cnt = idx.knn_with_ef_batch(base[:64], 5, 100)
        books = np.concatenate([np.ascontiguousarray(base[:16, lo:hi]).reshape(-1) for lo, hi in V.pq_groups(32, 8)])
        pq = V.PQTable(idx.vec_set, V.PQConfig(4, 8, "l2sqr"), books)
        pi, pd, pc = idx.knn_pq_batch(base[:64], 5, 100, pq)
        np.savez(sys.argv[1], links=idx.level0_links()[0], lens=idx.level0_links()[1], ids=ids, dd=dd, cnt=cnt, pi=pi,
                 pd=pd, pc=pc)
    """ % os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    out = {}
    for slots in ("", "64"):
        env = dict(os.environ)
        env.pop("VDB_HNSW_HASH_SLOTS", None)
        if slots:
            env["VDB_HNSW_HASH_SLOTS"] = slots
        path = str(tmp_path / f"run{slots}.npz")
        r = subprocess.run([sys.executable, "-c", code, path], capture_output=True, text=True, timeout=300, env=env)
        assert r.returncode == 0, r.stdout + r.stderr
        out[slots] = np.load(path)
    a, b = out[""], out["64"]
    assert (a["lens"] == b["lens"]).all()
    # entries past a list's length are never read (a re-run select may leave a longer first attempt's tail there)
    assert all((a["links"][i, :c] == b["links"][i, :c]).all() for i, c in enumerate(a["lens"]))
    for key in ("ids", "cnt", "pi", "pc"):
        assert (a[key] == b[key]).all(), key
    for key in ("dd", "pd"):
        assert (a[key].view(np.uint32) == b[key].view(np.uint32)).all(), key


def test_append_leaves_the_index_intact_when_it_fails(V):
    """vdb_hnsw_append builds the grown graph aside and swaps it in only on success (a failed cudaMalloc must not
    leave the handle with dangling or null arrays): a rejected append - here a bad level table - keeps the old graph
    searchable and bit-identical."""
    rng = np.random.default_rng(23)
    base = rng.random((4000, 24), dtype=np.float32)
    vs = V.DeviceVecSet(base[:3000], "l2sqr")
    idx = V.HNSWIndex(vs, V.HNSWConfig(0, 60, 8), rng=np.random.default_rng(2))
    before = idx.knn_with_ef_batch(base[:16], 5, 50)
    l0 = idx.level0_links()
    vs.push(base[3000:])
    bad = np.full(1000, 200, np.uint32)                        # level 200 is out of range: hnsw_alloc rejects it
    rc = V.lib().vdb_hnsw_append(idx._h, vs._h, V._lib.ptr(bad), 256)
    assert rc != 0
    n = V._lib.C.c_uint64(0)
    V._lib.check(V.lib().vdb_hnsw_info(idx._h, V._lib.C.byref(n), None, None, None, None))
    assert n.value == 3000                                     # the handle still describes the old graph
    links = np.zeros((3000, 16), np.uint32); lens = np.zeros(3000, np.uint32)
    V._lib.check(V.lib().vdb_hnsw_links0(idx._h, V._lib.ptr(links), V._lib.ptr(lens)))
    assert (links == l0[0]).all() and (lens == l0[1]).all()
    good = V.hnsw_rand_levels(1000, 8, np.random.default_rng(4))
    V._lib.check(V.lib().vdb_hnsw_append(idx._h, vs._h, V._lib.ptr(good), 256))   # and a proper append still works
    V._lib.check(V.lib().vdb_hnsw_info(idx._h, V._lib.C.byref(n), None, None, None, None))
    assert n.value == 4000


def test_evaluation_counter_counts_the_rows_a_search_gathers(V, fixtures):
    """vdb_hnsw_evals (the roofline unit of the HNSW bench legs): more rows are evaluated for a larger ef, never more
    than the graph holds per query, and the counter resets."""
    import ctypes as C
    from lab_1806_vec_db_b200 import _lib as L
    base, test = fixtures["base"], fixtures["test"][:64]
    vs = V.DeviceVecSet(base, "l2sqr")
    idx = V.HNSWIndex(vs, V.HNSWConfig(0, 100, 8), rng=np.random.default_rng(3))
    lib = L.lib()
    n = C.c_uint64(0)
    L.check(lib.vdb_hnsw_evals(idx._h, C.byref(n), 1))
    assert n.value > len(base)            # the build's own searches
    counts = []
    for ef in (10, 80):
        idx.knn_with_ef_batch(test, 10, ef)
        L.check(lib.vdb_hnsw_evals(idx._h, C.byref(n), 1))
        counts.append(n.value)
    assert 64 * 10 <= counts[0] < counts[1] <= 64 * len(base)
    L.check(lib.vdb_hnsw_evals(idx._h, C.byref(n), 0))
    assert n.value == 0
