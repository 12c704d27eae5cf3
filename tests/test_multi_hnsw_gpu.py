"""HNSW on a row-sharded set (vdb_init with several devices; csrc/multi.cu): one replica of the rows and the graph per
shard entry, every search one C call whose batch is split over the replicas.

Each query is walked by the single-GPU kernel on the same graph, so every result must be BIT-identical (ids, distance
bits, counts) to the unsharded index. The unsharded comparison index is loaded from the sharded index's own graph
(formats.hnsw_index_record -> HNSWIndex.from_record), so the comparison does not depend on whether the batched build is
deterministic. Runs on ONE GPU with three replicas on device 0, and with one replica per GPU when several are visible.
"""
import ctypes as C
import threading

import numpy as np
import pytest

from lab_1806_vec_db_b200 import formats as F

pytestmark = pytest.mark.gpu

M, EFC = 16, 100


def _data(n, nq, dim, seed=0, dtype=np.float32):
    rng = np.random.default_rng(seed)
    proto = rng.random((64, dim), dtype=np.float32)
    base = (proto[rng.integers(0, 64, n)] + 0.1 * rng.standard_normal((n, dim), dtype=np.float32)).clip(0, 1)
    q = (proto[rng.integers(0, 64, nq)] + 0.1 * rng.standard_normal((nq, dim), dtype=np.float32)).clip(0, 1)
    if dtype == np.uint8:
        return (base * 255).astype(np.uint8), (q * 255).astype(np.uint8)
    return base.astype(np.float32), q.astype(np.float32)


def _device_sets():
    import torch
    sets = [[0, 0, 0]]
    if torch.cuda.device_count() >= 2:
        sets.append(list(range(torch.cuda.device_count())))
    return sets


@pytest.fixture()
def vdb():
    import lab_1806_vec_db_b200 as V
    yield V
    V.init_devices([])


def _same(got, want):
    assert got[0].shape == want[0].shape
    assert (got[0].astype(np.int64) == want[0].astype(np.int64)).all()
    assert (np.asarray(got[1]).view(np.uint32) == np.asarray(want[1]).view(np.uint32)).all()
    assert (np.asarray(got[2]) == np.asarray(want[2])).all()


def _rows(x, lo, hi):
    return tuple(a[lo:hi] for a in x)


def _pair(V, base, metric, devs, levels):
    """(sharded index over `devs`, unsharded index loaded from the sharded index's graph, unsharded set)."""
    V.init_devices([])
    full_vs = V.DeviceVecSet(base, metric)
    V.init_devices(devs)
    vs = V.DeviceVecSet(base, metric)
    assert [d for d, _, _ in vs.shards()] == devs
    idx = V.HNSWIndex(vs, V.HNSWConfig(0, EFC, M), levels=levels)
    ref = V.HNSWIndex.from_record(full_vs, F.hnsw_index_record(idx))
    return idx, ref, full_vs


def _evals(V, idx, reset=1):
    n = C.c_uint64(0)
    V._lib.check(V.lib().vdb_hnsw_evals(idx._h, C.byref(n), reset))
    return n.value


@pytest.mark.parametrize("metric,dtype", [("l2sqr", np.float32), ("cosine", np.float32), ("l2sqr", np.uint8)])
def test_knn_with_ef_equals_the_unsharded_index(vdb, metric, dtype):
    V = vdb
    n, nq, dim = 20_000, 1000, 64
    base, q = _data(n, nq, dim, 1, dtype)
    levels = V.hnsw_rand_levels(n, M, np.random.default_rng(2))
    for devs in _device_sets():
        idx, ref, _ = _pair(V, base, metric, devs, levels)
        assert len(idx) == n and idx.enter_point == ref.enter_point
        # ef 1000 runs with the visited set in global memory
        for ef in (10, 100, 1000):
            for k in (1, 10, ef + 7):
                want = ref.knn_with_ef_batch(q, k, ef)
                _same(idx.knn_with_ef_batch(q, k, ef), want)
                for cnt in (0, 1, 2, 5):         # fewer queries than replicas, and a split into uneven slices
                    _same(idx.knn_with_ef_batch(q[:cnt], k, ef), _rows(want, 0, cnt))
        ids, dist, counts = idx.knn_with_ef_batch(q[:7], 0, 50)
        assert ids.shape == (7, 0) and (counts == 0).all()
        # the evaluation counters of the replicas add up to the unsharded count of the same batch
        _evals(V, idx), _evals(V, ref)
        _same(idx.knn_with_ef_batch(q, 10, 100), ref.knn_with_ef_batch(q, 10, 100))
        assert _evals(V, idx) == _evals(V, ref) > 0
        del idx, ref


def test_sequential_build_equals_the_unsharded_build_link_for_link(vdb, fixtures):
    """With one node per insertion batch the build is the reference's `add` path: the sharded build (on replica 0) must
    produce the unsharded build's graph exactly, and every replica holds that graph."""
    V = vdb
    base = fixtures["base"]
    levels = V.hnsw_rand_levels(len(base), 8, np.random.default_rng(4))
    old = V.HNSWIndex.MAX_BATCH
    try:
        V.HNSWIndex.MAX_BATCH = 1
        V.init_devices([])
        one = V.HNSWIndex(V.DeviceVecSet(base, "l2sqr"), V.HNSWConfig(0, 60, 8), levels=levels)
        for devs in _device_sets():
            V.init_devices(devs)
            sh = V.HNSWIndex(V.DeviceVecSet(base, "l2sqr"), V.HNSWConfig(0, 60, 8), levels=levels)
            a, b = one.level0_links(), sh.level0_links()
            assert (a[1] == b[1]).all() and (a[0] == b[0]).all()
            assert one.enter_point == sh.enter_point
            assert all((x == y).all() for x, y in zip(one.upper_links(), sh.upper_links()))
            q = fixtures["test"][:50]
            _same(sh.knn_with_ef_batch(q, 10, 40), one.knn_with_ef_batch(q, 10, 40))
            del sh
    finally:
        V.HNSWIndex.MAX_BATCH = old


def test_single_queries_rotate_over_the_replicas(vdb):
    V = vdb
    n, nq, dim = 8_000, 64, 32
    base, q = _data(n, nq, dim, 3)
    levels = V.hnsw_rand_levels(n, M, np.random.default_rng(3))
    for devs in _device_sets():
        idx, ref, _ = _pair(V, base, "l2sqr", devs, levels)
        want = idx.knn_with_ef_batch(q, 10, 64)
        _same(want, ref.knn_with_ef_batch(q, 10, 64))
        for i in range(len(devs) + 1):           # every replica serves at least one of these calls
            _same(idx.knn_with_ef_batch(q[i:i + 1], 10, 64), _rows(want, i, i + 1))
            assert [p.index for p in idx.knn_with_ef(q[i], 10, 64)] == want[0][i].tolist()
        # a graph loaded onto the sharded set (vdb_hnsw_create_from_graph) is replicated the same way
        back = V.HNSWIndex.from_record(idx.vec_set, F.hnsw_index_record(idx))
        _same(back.knn_with_ef_batch(q, 10, 64), want)
        _same(back.knn_with_ef_batch(q[5:6], 10, 64), _rows(want, 5, 6))
        del idx, ref, back


def test_concurrent_single_and_batched_calls(vdb):
    """The HNSW calls are re-entrant: six threads mix single-query and batched calls on one sharded index."""
    V = vdb
    n, nq, dim = 8_000, 96, 32
    base, q = _data(n, nq, dim, 4)
    levels = V.hnsw_rand_levels(n, M, np.random.default_rng(4))
    idx, ref, _ = _pair(V, base, "l2sqr", [0, 0, 0], levels)
    want = ref.knn_with_ef_batch(q, 10, 80)
    errs, outs = [], [None] * 6

    def work(i):
        try:
            got = []
            for r in range(4):
                got.append(("batch", idx.knn_with_ef_batch(q, 10, 80)))
                j = (i * 7 + r) % nq
                got.append((j, idx.knn_with_ef_batch(q[j:j + 1], 10, 80)))
            outs[i] = got
        except Exception as e:  # noqa: BLE001
            errs.append(e)

    th = [threading.Thread(target=work, args=(i,)) for i in range(6)]
    [t.start() for t in th]
    [t.join() for t in th]
    assert not errs, errs
    for got in outs:
        for tag, res in got:
            _same(res, want if tag == "batch" else _rows(want, tag, tag + 1))


def _books(V, base, dim, m, n_bits, at=100):
    kc = 1 << n_bits
    return np.concatenate([np.ascontiguousarray(base[at:at + kc, lo:hi]).reshape(-1) for lo, hi in V.pq_groups(dim, m)])


@pytest.mark.parametrize("metric", ["l2sqr", "cosine"])
def test_knn_pq_equals_the_unsharded_index(vdb, metric):
    """A 4-bit table built on the sharded set is searched through an unsharded copy of it on every replica: identical to
    an unsharded table with the same codebooks, on the same graph."""
    V = vdb
    n, nq, dim, m = 20_000, 300, 64, 16
    base, q = _data(n, nq, dim, 5)
    levels = V.hnsw_rand_levels(n, M, np.random.default_rng(5))
    books_a, books_b = _books(V, base, dim, m, 4, 100), _books(V, base, dim, m, 4, 5000)
    for devs in _device_sets():
        idx, ref, full_vs = _pair(V, base, metric, devs, levels)
        full_a = V.PQTable(full_vs, V.PQConfig(4, m, metric), books_a)
        full_b = V.PQTable(full_vs, V.PQConfig(4, m, metric), books_b)
        pq_a = V.PQTable(idx.vec_set, V.PQConfig(4, m, metric), books_a)
        pq_b = V.PQTable(idx.vec_set, V.PQConfig(4, m, metric), books_b)
        want_a = {(k, ef): ref.knn_pq_batch(q, k, ef, full_a) for k, ef in ((10, 20), (10, 100), (50, 30))}
        want_b = ref.knn_pq_batch(q, 10, 100, full_b)
        for (k, ef), w in want_a.items():
            _same(idx.knn_pq_batch(q, k, ef, pq_a), w)
            _same(idx.knn_pq_batch(q[:2], k, ef, pq_a), _rows(w, 0, 2))
        for _ in range(2):                       # alternating tables: each call gets its own table's results
            _same(idx.knn_pq_batch(q, 10, 100, pq_b), want_b)
            _same(idx.knn_pq_batch(q, 10, 100, pq_a), want_a[(10, 100)])
        assert [p.index for p in idx.knn_pq(q[3], 10, 100, pq_b)] == want_b[0][3].tolist()
        # tables of another set: an unsharded table, a table of another sharded set
        with pytest.raises(V.VdbError) as e:
            idx.knn_pq_batch(q, 10, 100, full_a)
        assert e.value.code == V._lib.EINVAL
        other_vs = V.DeviceVecSet(base, metric)
        other = V.PQTable(other_vs, V.PQConfig(4, m, metric), books_a)
        with pytest.raises(V.VdbError) as e:
            idx.knn_pq_batch(q, 10, 100, other)
        assert e.value.code == V._lib.EINVAL
        # 8-bit tables keep the HNSW + PQ refusal
        pq8 = V.PQTable(idx.vec_set, V.PQConfig(8, m, metric), _books(V, base, dim, m, 8))
        with pytest.raises(V.VdbError, match="4-bit"):
            idx.knn_pq_batch(q, 10, 100, pq8)
        _same(idx.knn_pq_batch(q, 10, 100, pq_a), want_a[(10, 100)])
        del idx, ref, pq_a, pq_b, pq8, other, other_vs


def test_sets_and_tables_of_another_metric_are_refused(vdb):
    V = vdb
    L = V._lib
    base, q = _data(3_000, 8, 32, 6)
    levels = V.hnsw_rand_levels(3_000, M, np.random.default_rng(6))
    V.init_devices([0, 0, 0])
    vs_l2 = V.DeviceVecSet(base, "l2sqr")
    vs_cos = V.DeviceVecSet(base, "cosine")
    idx = V.HNSWIndex(vs_l2, V.HNSWConfig(0, EFC, M), levels=levels)
    pq_cos = V.PQTable(vs_cos, V.PQConfig(4, 8, "cosine"), _books(V, base, 32, 8, 4))
    ids, dist, cnt = np.zeros((8, 10), np.uint64), np.zeros((8, 10), np.float32), np.zeros(8, np.uint32)
    out = (L.ptr(ids), L.ptr(dist), L.ptr(cnt))
    assert V.lib().vdb_hnsw_knn_pq(vs_l2._h, idx._h, pq_cos._h, L.ptr(q), 8, 10, 20, *out) == L.EINVAL
    assert V.lib().vdb_hnsw_knn(vs_cos._h, idx._h, L.ptr(q), 8, 10, 20, *out) == L.EINVAL


def test_fewer_rows_than_replicas(vdb):
    V = vdb
    rng = np.random.default_rng(7)
    base, q = rng.random((2, 12), dtype=np.float32), rng.random((6, 12), dtype=np.float32)
    levels = np.array([1, 0], np.uint32)
    idx, ref, _ = _pair(V, base, "l2sqr", [0, 0, 0, 0], levels)
    assert [h - lo for _, lo, h in idx.vec_set.shards()] == [1, 1, 0, 0]
    for k in (1, 2, 5):
        want = ref.knn_with_ef_batch(q, k, 10)
        _same(idx.knn_with_ef_batch(q, k, 10), want)
        assert (want[2] == min(k, 2)).all()


def test_refusals_destroy_and_rebuild(vdb):
    V = vdb
    L = V._lib
    lib = V.lib()
    n, dim = 4_000, 32
    base, q = _data(n, 16, dim, 8)
    levels = V.hnsw_rand_levels(n, M, np.random.default_rng(8))
    V.init_devices([])
    plain_vs = V.DeviceVecSet(base, "l2sqr")
    plain = V.HNSWIndex(plain_vs, V.HNSWConfig(0, EFC, M), levels=levels)
    V.init_devices([0, 0, 0])
    vs = V.DeviceVecSet(base, "l2sqr")
    vs2 = V.DeviceVecSet(base, "l2sqr")
    idx = V.HNSWIndex(vs, V.HNSWConfig(0, EFC, M), levels=levels)
    want = idx.knn_with_ef_batch(q, 10, 50)
    ids = np.zeros((16, 10), np.uint64)
    dist = np.zeros((16, 10), np.float32)
    cnt = np.zeros(16, np.uint32)
    # an index built on an unsharded set with the same rows, or on another sharded set
    assert lib.vdb_hnsw_knn(vs._h, plain._h, L.ptr(q), 16, 10, 50, L.ptr(ids), L.ptr(dist), L.ptr(cnt)) == L.EINVAL
    assert lib.vdb_hnsw_knn(vs2._h, idx._h, L.ptr(q), 16, 10, 50, L.ptr(ids), L.ptr(dist), L.ptr(cnt)) == L.EINVAL
    # the replicated index on an unsharded set
    assert lib.vdb_hnsw_knn(plain_vs._h, idx._h, L.ptr(q), 16, 10, 50, L.ptr(ids), L.ptr(dist), L.ptr(cnt)) == L.EINVAL
    # device-pointer variants and appends have no row-sharded implementation
    assert lib.vdb_hnsw_knn_dev(vs._h, idx._h, None, 0, 10, 50, None, None, None, None) == L.EUNSUPPORTED
    pq = V.PQTable(vs, V.PQConfig(4, 8, "l2sqr"), _books(V, base, dim, 8, 4))
    assert lib.vdb_hnsw_knn_pq_dev(vs._h, idx._h, pq._h, None, 0, 10, 50, None, None, None, None) == L.EUNSUPPORTED
    lv = np.zeros(1, np.uint32)
    assert lib.vdb_hnsw_append(idx._h, vs._h, L.ptr(lv), 1) == L.EUNSUPPORTED
    assert lib.vdb_hnsw_append(idx._h, plain_vs._h, L.ptr(lv), 1) == L.EUNSUPPORTED
    ov = C.c_uint32(1)
    L.check(lib.vdb_hnsw_overflow(idx._h, C.byref(ov)))
    assert ov.value == 0
    _same(idx.knn_with_ef_batch(q, 10, 50), want)            # the refusals left the index intact
    idx.close()
    del pq, vs, vs2
    V.init_devices([])
    V.init_devices([0, 0])
    vs3 = V.DeviceVecSet(base, "l2sqr")
    again = V.HNSWIndex(vs3, V.HNSWConfig(0, EFC, M), levels=levels)
    ref = V.HNSWIndex.from_record(plain_vs, F.hnsw_index_record(again))
    _same(again.knn_with_ef_batch(q, 10, 50), ref.knn_with_ef_batch(q, 10, 50))


def test_gist_1000_recall_matches_the_unsharded_index(vdb, fixtures, oracle):
    V = vdb
    base, test = fixtures["base"], fixtures["test"][:200]
    levels = V.hnsw_rand_levels(len(base), M, np.random.default_rng(5))
    gt = oracle.flat_knn(base, test, 10, "l2sqr", nthreads=8)[0]

    def recall(ids):
        return float(np.mean([len(set(a.tolist()) & set(b.tolist())) / len(b) for a, b in zip(ids, gt)]))

    for devs in _device_sets():
        idx, ref, _ = _pair(V, base, "l2sqr", devs, levels)
        for ef in (10, 50, 100):
            got, want = idx.knn_with_ef_batch(test, 10, ef), ref.knn_with_ef_batch(test, 10, ef)
            _same(got, want)
            assert recall(got[0]) == recall(want[0])
        assert recall(idx.knn_with_ef_batch(test, 10, 100)[0]) >= 0.99
        del idx, ref
