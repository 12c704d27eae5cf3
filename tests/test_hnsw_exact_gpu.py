"""HNSW kernels bit for bit against the CPU restatement, on data where every distance is exact (test_hnsw_exact_cpu.py):
integer rows, queries and codebooks below the 2^24 bound. The device and the oracle then compute the same distance
bits in any summation order, so

- a search over the same graph (the device's, exported and walked by HnswOracle.from_graph) returns the same ids and
  the same distance bits for every query on which the oracle met no tie event; the few queries that met one pass the
  tolerance rule of assert_knn_parity, and each case prints how many there were;
- a build on data where the oracle met no tie event gives the oracle's graph list for list: MAX_BATCH = 1 against
  the sequential build, larger batches against the restated batch pipeline (orc_hnsw_build_batched).

A kernel that drops one candidate, breaks the search one step early or late, reads a row short, or orders a batch's
links differently changes a few lists or a few results: these tests count every one of them."""
import ctypes as C

import numpy as np
import pytest

from conftest import assert_knn_parity
from test_hnsw_exact_cpu import assert_exact, differing_lists, exact_rows, oracle_graph

pytestmark = pytest.mark.gpu

K = 10
EFS = (1, K, 100, 448, 449, 640, 641, 896, 897, 4096)   # every visited-set tier edge of hash_cap_for, and ef > n


@pytest.fixture(scope="module")
def V():
    import lab_1806_vec_db_b200 as V
    return V


def _rows(rng, n, dim, dtype):
    """exact rows: the largest magnitude the 2^24 bound allows at this dim (signed f32, unsigned u8)"""
    r = int(np.sqrt((2 ** 24 - 1) / (2 * dim)))
    if dtype == np.uint8:
        return exact_rows(rng, n, dim, np.uint8, 0, min(r, 255))
    return exact_rows(rng, n, dim, np.float32, -min(r, 1000), min(r, 1000))


def _build(V, base, metric, M, efc, levels, max_batch=None):
    old = V.HNSWIndex.MAX_BATCH
    if max_batch is not None:
        V.HNSWIndex.MAX_BATCH = max_batch
    try:
        return V.HNSWIndex(V.DeviceVecSet(base, metric), V.HNSWConfig(0, efc, M), levels=levels)
    finally:
        V.HNSWIndex.MAX_BATCH = old


def _device_graph(idx):
    links0, len0 = idx.level0_links()
    _, ulinks, ulen = idx.upper_links()
    return links0, len0, ulinks, ulen


def _oracle_on(idx, base, metric, M, efc):
    from oracle.oracle_py import HnswOracle
    links0, len0, ulinks, ulen = _device_graph(idx)
    ep, el = idx.enter_point
    return HnswOracle.from_graph(base, metric, M, efc, idx.levels, links0, len0, ulinks, ulen, ep, el)


def _overflow(V, idx):
    ov = C.c_uint32(7)
    V._lib.check(V.lib().vdb_hnsw_overflow(idx._h, C.byref(ov)))
    return ov.value


def check_same(tag, base, queries, metric, got, want, oracle):
    """ids and distance bits equal on every query without a tie event; the others by assert_knn_parity. Returns the
    number of tie-excused queries."""
    gi, gd, gc = got
    wi, wd, wc, ties = want
    assert gi.shape == wi.shape and (gc == wc).all(), f"{tag}: result counts differ"
    clean = np.nonzero(ties == 0)[0]
    for q in clean:
        c = int(wc[q])
        assert (gi[q, :c] == wi[q, :c]).all(), f"{tag}: query {q}: ids {gi[q, :c]} vs {wi[q, :c]}"
        assert (gd[q, :c].view(np.uint32) == wd[q, :c].view(np.uint32)).all(), (
            f"{tag}: query {q}: distance bits {gd[q, :c]} vs {wd[q, :c]}")
    tied = np.nonzero(ties)[0]
    if tied.size:
        assert_knn_parity(base, queries[tied], metric, (gi[tied], gd[tied], gc[tied]), (wi[tied], wd[tied], wc[tied]),
                          oracle)
    print(f"{tag}: {tied.size} of {len(ties)} queries excused by tie events")
    return int(tied.size)


# (dtype, metric, dim, M): every non-PQ instantiation of hnsw_search_kernel, row lengths on both sides of the 1024-element
# chunk of warp_dot_row (and two chunks), M = 2 (deep graphs) to M = 32 (64-link lists, two 32-wide rounds per expansion)
SEARCH_CASES = [
    (np.float32, "l2sqr", 2, 2), (np.float32, "l2sqr", 3, 8), (np.float32, "l2sqr", 17, 32), (np.float32, "l2sqr", 64, 8),
    (np.float32, "l2sqr", 1023, 8), (np.float32, "l2sqr", 1024, 2), (np.float32, "l2sqr", 1025, 8),
    (np.float32, "l2sqr", 2050, 32),
    (np.float32, "cosine", 3, 8), (np.float32, "cosine", 64, 32), (np.float32, "cosine", 1025, 2),
    (np.float32, "cosine", 2050, 8),
    (np.uint8, "l2sqr", 15, 8), (np.uint8, "l2sqr", 16, 2), (np.uint8, "l2sqr", 17, 32), (np.uint8, "l2sqr", 100, 8),
    (np.uint8, "l2sqr", 1025, 8), (np.uint8, "l2sqr", 2050, 2),
    (np.uint8, "cosine", 16, 8), (np.uint8, "cosine", 100, 32), (np.uint8, "cosine", 2050, 8),
]


@pytest.mark.parametrize("dtype,metric,dim,M", SEARCH_CASES,
                         ids=[f"{np.dtype(c[0]).name}-{c[1]}-d{c[2]}-M{c[3]}" for c in SEARCH_CASES])
def test_search_on_the_same_graph_is_bit_exact(V, oracle, dtype, metric, dim, M):
    rng = np.random.default_rng(dim * 131 + M)
    n, nq, efc = 3000, 120, 100
    base, q = _rows(rng, n, dim, dtype), _rows(rng, nq, dim, dtype)
    assert_exact(base, q)
    levels = V.hnsw_rand_levels(n, M, rng)
    idx = _build(V, base, metric, M, efc, levels)
    cpu = _oracle_on(idx, base, metric, M, efc)
    tied = 0
    for ef in EFS:
        got = idx.knn_with_ef_batch(q, K, ef)
        want = cpu.knn(q, K, ef, nthreads=oracle.ncores(), ties=True)
        tied += check_same(f"ef {ef}", base, q, metric, got, want, oracle)
    assert _overflow(V, idx) == 0
    assert tied <= len(EFS) * nq // 20, tied


def test_search_edges_k_ef_n_and_batch_sizes(V, oracle):
    """k > ef (ef becomes k), ef > n, k > n, k = 0, and 0, 1 and 1000 queries"""
    rng = np.random.default_rng(77)
    n, dim, M, efc = 2500, 64, 8, 60
    base = _rows(rng, n, dim, np.float32)
    q = _rows(rng, 1000, dim, np.float32)
    idx = _build(V, base, "l2sqr", M, efc, V.hnsw_rand_levels(n, M, rng))
    cpu = _oracle_on(idx, base, "l2sqr", M, efc)
    for nq, k, ef in ((1000, K, 50), (1, K, 50), (1, 1, 1), (200, 30, 5), (100, 40, 3000)):
        got = idx.knn_with_ef_batch(q[:nq], k, ef)
        check_same(f"nq {nq} k {k} ef {ef}", base, q[:nq], "l2sqr", got,
                   cpu.knn(q[:nq], k, ef, nthreads=oracle.ncores(), ties=True), oracle)
    ids, dd, cnt = idx.knn_with_ef_batch(q[:0], K, 50)
    assert ids.shape == (0, K) and cnt.shape == (0,)
    ids, dd, cnt = idx.knn_with_ef_batch(q[:7], 0, 50)
    assert ids.shape == (7, 0) and (cnt == 0).all()
    # k > n on a small set: every row, in order
    small = base[:40]
    si = _build(V, small, "l2sqr", 4, 20, V.hnsw_rand_levels(40, 4, rng))
    scpu = _oracle_on(si, small, "l2sqr", 4, 20)
    got = si.knn_with_ef_batch(q[:20], 64, 10)
    assert (got[2] == 40).all()
    check_same("k > n", small, q[:20], "l2sqr", got, scpu.knn(q[:20], 64, 10, ties=True), oracle)
    assert _overflow(V, idx) == 0 and _overflow(V, si) == 0


# (row dtype, metric, dim, m): the two PQ instantiations over f32 and u8 rows; m odd, m > 32 (two lanes' rounds), m = dim
PQ_CASES = [
    (np.float32, "l2sqr", 64, 7), (np.float32, "cosine", 96, 48), (np.uint8, "l2sqr", 40, 40), (np.uint8, "cosine", 66, 33),
    (np.float32, "l2sqr", 70, 35), (np.uint8, "cosine", 128, 64),
]


@pytest.mark.parametrize("dtype,metric,dim,m", PQ_CASES,
                         ids=[f"{np.dtype(c[0]).name}-{c[1]}-d{c[2]}-m{c[3]}" for c in PQ_CASES])
def test_pq_search_on_the_same_graph_is_bit_exact(V, oracle, dtype, metric, dim, m):
    rng = np.random.default_rng(dim * 7 + m)
    n, nq, M, efc = 3000, 100, 8, 80
    r = int(np.sqrt((2 ** 24 - 1) / (4 * dim))) if dtype == np.float32 else 255
    base = (exact_rows(rng, n, dim, dtype, -r, r) if dtype == np.float32 else exact_rows(rng, n, dim, dtype, 0, 255))
    q = base[rng.integers(0, n, nq)] if dtype == np.uint8 else exact_rows(rng, nq, dim, dtype, -r, r)
    books = np.concatenate([np.ascontiguousarray(base[200:216, lo:hi]).reshape(-1) for lo, hi in V.pq_groups(dim, m)])
    assert_exact(base, q, books, pq_l2=metric == "l2sqr")
    vs = V.DeviceVecSet(base, metric)
    pq = V.PQTable(vs, V.PQConfig(4, m, metric), books)
    idx = V.HNSWIndex(vs, V.HNSWConfig(0, efc, M), levels=V.hnsw_rand_levels(n, M, rng))
    cpu = _oracle_on(idx, base, metric, M, efc)
    for ef in (1, K, 100, 449, 897, 4096):
        got = idx.knn_pq_batch(q, K, ef, pq)
        want = cpu.knn_pq(q, K, ef, pq.encoded_vec_set, books, m, 4, nthreads=oracle.ncores(), ties=True)
        check_same(f"pq ef {ef}", base, q, metric, got, want, oracle)
    assert _overflow(V, idx) == 0


def test_device_entry_points_give_the_host_calls_bits(V):
    """vdb_hnsw_knn_dev / vdb_hnsw_knn_pq_dev on device queries: the bits of the host calls"""
    import torch
    V.init_devices([])
    lib, L = V.lib(), V._lib
    rng = np.random.default_rng(8)
    n, nq, dim, m, M = 2000, 64, 48, 12, 8
    base, q = _rows(rng, n, dim, np.float32), _rows(rng, nq, dim, np.float32)
    vs = V.DeviceVecSet(base, "cosine")
    books = np.concatenate([np.ascontiguousarray(base[:16, lo:hi]).reshape(-1) for lo, hi in V.pq_groups(dim, m)])
    pq = V.PQTable(vs, V.PQConfig(4, m, "cosine"), books)
    idx = V.HNSWIndex(vs, V.HNSWConfig(0, 60, M), levels=V.hnsw_rand_levels(n, M, rng))
    qd = torch.from_numpy(q).cuda()
    p = lambda t: C.c_void_p(t.data_ptr())
    for ef in (20, 900):
        for host, call in ((idx.knn_with_ef_batch(q, K, ef),
                            lambda i, d, c: lib.vdb_hnsw_knn_dev(vs._h, idx._h, p(qd), nq, K, ef, i, d, c, None)),
                           (idx.knn_pq_batch(q, K, ef, pq),
                            lambda i, d, c: lib.vdb_hnsw_knn_pq_dev(vs._h, idx._h, pq._h, p(qd), nq, K, ef, i, d, c, None))):
            ids = torch.zeros((nq, K), dtype=torch.int64, device="cuda")
            dd = torch.zeros((nq, K), dtype=torch.float32, device="cuda")
            cnt = torch.zeros((nq,), dtype=torch.int32, device="cuda")
            L.check(call(p(ids), p(dd), p(cnt)))
            torch.cuda.synchronize()
            assert (cnt.cpu().numpy() == host[2]).all()
            assert (ids.cpu().numpy().view(np.uint64) == host[0]).all()
            assert (dd.cpu().numpy().view(np.uint32) == host[1].view(np.uint32)).all()
    assert _overflow(V, idx) == 0


def _zero_tie_build(V, rng_seed, dtype, metric, dim, M, efc, n, max_batch, n0=0):
    """levels and rows on which the oracle's build meets no tie event (first of a few seeds), and that oracle graph"""
    from oracle.oracle_py import HnswOracle
    for s in range(10):
        rng = np.random.default_rng(rng_seed + 1000 * s)
        base = _rows(rng, n, dim, dtype)
        assert_exact(base)
        levels = V.hnsw_rand_levels(n, M, rng)
        if max_batch == 1 and n0 == 0:
            ref = HnswOracle(base, metric, M, efc, levels)
        else:
            ref = HnswOracle.batched(base, metric, M, efc, levels, max_batch, n0)
        if ref.build_ties == 0:
            return base, levels, ref
        print(f"seed {s}: {ref.build_ties} build tie events, next seed")
    pytest.fail("no seed without build tie events")


# (dtype, metric, dim, M, max_batch, n): MAX_BATCH = 1 is the sequential build; 7, 64 and 2048 the batched pipeline
# (M = 2 on 5000 rows reaches batches of 2048 once 4096 rows are in)
BUILD_CASES = [
    (np.float32, "l2sqr", 64, 8, 1, 1500), (np.uint8, "cosine", 64, 2, 1, 1500), (np.float32, "cosine", 3, 32, 1, 1200),
    (np.uint8, "l2sqr", 1025, 8, 1, 800),
    (np.float32, "l2sqr", 64, 8, 7, 3000), (np.float32, "cosine", 1025, 2, 7, 2000), (np.uint8, "cosine", 64, 32, 7, 3000),
    (np.float32, "l2sqr", 3, 2, 64, 4000), (np.uint8, "l2sqr", 64, 8, 64, 1500), (np.float32, "cosine", 64, 32, 64, 4000),
    (np.float32, "l2sqr", 64, 2, 2048, 5000), (np.uint8, "cosine", 64, 8, 2048, 5000),
    (np.float32, "l2sqr", 1025, 32, 2048, 3000), (np.float32, "cosine", 3, 8, 2048, 5000),
]


@pytest.mark.parametrize("dtype,metric,dim,M,max_batch,n", BUILD_CASES,
                         ids=[f"{np.dtype(c[0]).name}-{c[1]}-d{c[2]}-M{c[3]}-b{c[4]}-n{c[5]}" for c in BUILD_CASES])
def test_build_gives_the_oracle_graph_link_for_link(V, oracle, dtype, metric, dim, M, max_batch, n):
    efc = 40
    base, levels, ref = _zero_tie_build(V, dim * 17 + M * 3 + max_batch, dtype, metric, dim, M, efc, n, max_batch)
    idx = _build(V, base, metric, M, efc, levels, max_batch)
    bad = differing_lists(_device_graph(idx), oracle_graph(ref))
    print(f"{bad} differing adjacency lists of {n} rows, 0 build tie events")
    assert bad == 0
    assert idx.enter_point == ref.enter_point
    assert _overflow(V, idx) == 0


@pytest.mark.parametrize("dtype,metric,dim,M,max_batch", [
    (np.float32, "l2sqr", 64, 8, 1), (np.float32, "cosine", 1025, 8, 64), (np.float32, "l2sqr", 3, 2, 2048),
    (np.uint8, "cosine", 64, 32, 7),
])
def test_append_gives_the_oracle_graph_link_for_link(V, oracle, dtype, metric, dim, M, max_batch):
    """batch_add_pushed onto a built index: build(n0) + append(n - n0) with the same levels is the oracle's build of
    n0 rows followed by its append, batch sizes restarting at done = n0"""
    n, n0, efc = 3000, 1100, 40
    base, levels, ref = _zero_tie_build(V, dim + M + max_batch, dtype, metric, dim, M, efc, n, max_batch, n0)
    vs = V.DeviceVecSet(base[:n0], metric)
    old = V.HNSWIndex.MAX_BATCH
    V.HNSWIndex.MAX_BATCH = max_batch
    try:
        idx = V.HNSWIndex(vs, V.HNSWConfig(0, efc, M), levels=levels[:n0])
        vs.push(base[n0:])
        idx.batch_add_pushed(levels=levels[n0:])
    finally:
        V.HNSWIndex.MAX_BATCH = old
    bad = differing_lists(_device_graph(idx), oracle_graph(ref))
    print(f"{bad} differing adjacency lists of {n} rows after an append, 0 build tie events")
    assert bad == 0 and idx.enter_point == ref.enter_point


@pytest.mark.parametrize("M", [16, 32])
def test_visited_set_room_on_large_hard_sets(V, oracle, M):
    """50 000 uniform rows of dim 64: the walks evaluate more distinct rows than 7/8 of the smallest shared-memory
    visited set holds (8192 slots up to ef 448). Every build and search must succeed, and on the same graph give the
    oracle's results (float data: by the tolerance rule, ties within it excused)."""
    rng = np.random.default_rng(50 + M)
    n, dim, nq = 50_000, 64, 50
    base = rng.random((n, dim), dtype=np.float32)
    q = rng.random((nq, dim), dtype=np.float32)
    vs = V.DeviceVecSet(base, "l2sqr")
    for efc in (200, 448):
        idx = V.HNSWIndex(vs, V.HNSWConfig(0, efc, M), rng=np.random.default_rng(efc))
        cpu = _oracle_on(idx, base, "l2sqr", M, efc)
        for ef in (448, 640, 896):
            got = idx.knn_with_ef_batch(q, K, ef)
            want = cpu.knn(q, K, ef, nthreads=oracle.ncores())
            rate = assert_knn_parity(base, q, "l2sqr", got, want, oracle)
            print(f"M {M} efc {efc} ef {ef}: exact-id rate {rate:.4f}")
            assert rate >= 0.99
        assert _overflow(V, idx) == 0
