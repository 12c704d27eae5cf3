"""Flat kNN for any k: the large-k path (csrc/topk_large.cu and the emit instantiation of the scan, csrc/flat_scan.cu).

The reference's FlatIndex::knn takes any k (a BTreeSet result set, src/index_algorithm/flat_index.rs:48-57) and returns
min(k, n) rows; VecDB.search asks for k = len(table) to mean "every row within upper_bound". Above the k that the fused
shared-memory top-k holds, every entry point takes the select + sort path in global memory. Its first k_fused columns
must be the fused call's bits: (distance, id) is a strict total order, so the top k' is a prefix of the top k.

Row-sharded cases run on one GPU with three virtual shards (init_devices([0, 0, 0])), and with one shard per GPU when
several are visible.
"""
import ctypes as C
import threading

import numpy as np
import pytest

from conftest import assert_knn_parity

pytestmark = pytest.mark.gpu

SMEM_MAX = 200 * 1024


def k_fused(dim, dtype, nq):
    """The largest k the fused top-k of the scan holds for a batch of nq queries (flat_scan.cu: scan_fit and
    merge_keys_fits): the scan's shared-memory segments, and the merge's when the per-CTA lists are merged."""
    vec = 4 if dtype == np.float32 else 16
    nvec = -(-dim // vec)
    nit = -(-nvec // 32)
    qbytes = nit * 32 * vec * 4 if dtype == np.float32 else nit * 32 * 16
    sync = lambda r: max(max(1, 64 // (8 * r)), -(-8 // nit))  # noqa: E731
    period = max(sync(4) * 8 * 4, sync(8) * 8 * 8)
    p2 = lambda v: 1 << max(0, (v - 1).bit_length())  # noqa: E731
    smem = lambda t, k: t * qbytes + t * p2(k + 2 * period) * 8 + t * 4  # noqa: E731

    def fits(k):
        t = 8
        while t > 1 and smem(t, k) > SMEM_MAX:
            t //= 2
        if smem(t, k) > SMEM_MAX:
            return False
        merged = not (nq <= 8 and nq <= t)
        return not merged or p2(k + 512) * 8 + 4 <= SMEM_MAX

    lo, hi = 1, 1 << 16
    while lo < hi:
        mid = (lo + hi + 1) // 2
        lo, hi = (mid, hi) if fits(mid) else (lo, mid - 1)
    return lo


def _data(n, nq, dim, seed, dtype):
    rng = np.random.default_rng(seed)
    proto = rng.random((64, dim), dtype=np.float32) * 0.2
    base = (proto[rng.integers(0, 64, n)] + 0.03 * rng.standard_normal((n, dim), dtype=np.float32)).clip(0, 1)
    q = (proto[rng.integers(0, 64, nq)] + 0.03 * rng.standard_normal((nq, dim), dtype=np.float32)).clip(0, 1)
    if dtype == np.uint8:
        return (base * 255).astype(np.uint8), (q * 255).astype(np.uint8)
    return base.astype(np.float32), q.astype(np.float32)


def _same(got, want, cols=None):
    c = slice(None) if cols is None else slice(0, cols)
    assert (got[0][:, c].astype(np.int64) == want[0][:, c].astype(np.int64)).all()
    assert (np.asarray(got[1])[:, c].view(np.uint32) == np.asarray(want[1])[:, c].view(np.uint32)).all()
    if cols is None:
        assert (np.asarray(got[2]) == np.asarray(want[2])).all()


def _check_structure(res, n, k):
    ids, dist, cnt = res
    m = min(k, n)
    assert ids.shape[1] == k and (cnt == m).all()
    assert (ids[:, m:] == np.iinfo(np.uint64).max).all() and np.isnan(dist[:, m:]).all()
    v_ids, v_d = ids[:, :m].astype(np.int64), dist[:, :m]
    assert (v_ids < n).all() and not np.isnan(v_d).any()
    # ascending by (distance, id)
    dd, di = np.diff(v_d.astype(np.float64), axis=1), np.diff(v_ids, axis=1)
    assert ((dd > 0) | ((dd == 0) & (di > 0))).all()
    for row in v_ids:
        assert len(np.unique(row)) == m
    if k >= n:
        assert (np.sort(v_ids, axis=1) == np.arange(n)).all()


@pytest.fixture()
def vdb():
    import lab_1806_vec_db_b200 as V
    yield V
    V.init_devices([])
    V._lib.check(V.lib().vdb_flat_set_path(0))


def _device_sets():
    import torch
    sets = [[0, 0, 0]]
    if torch.cuda.device_count() >= 2:
        sets.append(list(range(min(torch.cuda.device_count(), 4))))
    return sets


@pytest.mark.parametrize("metric,dtype", [("l2sqr", np.float32), ("cosine", np.float32), ("l2sqr", np.uint8),
                                          ("cosine", np.uint8)])
def test_any_k_is_a_prefix_extension_of_the_fused_call(vdb, oracle, metric, dtype):
    V = vdb
    V.init_devices([])
    n, dim = 100_000, 96
    base, q = _data(n, 17, dim, 1, dtype)
    idx = V.FlatIndex.from_vec_set(base, metric)
    for nq in (1, 3, 17):
        kf = k_fused(dim, dtype, nq)
        fused = idx.knn_batch(q[:nq], kf)
        _check_structure(fused, n, kf)
        prev = None
        for k in (kf + 1, 50_000, n, n + 7):
            got = idx.knn_batch(q[:nq], k)
            _check_structure(got, n, k)
            _same(got, fused, kf)
            if prev is not None:
                _same(got, prev, prev[0].shape[1] if prev[0].shape[1] <= n else n)
            prev = got
    # oracle parity at a large k on a few queries
    k = 50_000
    got = idx.knn_batch(q[:2], k)
    want = oracle.flat_knn(base, q[:2], k, metric, nthreads=8)
    assert_knn_parity(base, q[:2], metric, got, want, oracle)


def test_single_query_calls_bypass_the_batcher_and_match_serial_calls(vdb):
    V = vdb
    V.init_devices([])
    n, dim = 80_000, 64
    base, q = _data(n, 8, dim, 2, np.float32)
    idx = V.FlatIndex.from_vec_set(base, "l2sqr")
    lib = V.lib()
    k = 40_000
    serial = [idx.knn_batch(q[i:i + 1], k) for i in range(8)]
    b0, s0 = C.c_uint64(), C.c_uint64()
    V._lib.check(lib.vdb_batch_stats(idx.vec_set._h, C.byref(b0), C.byref(s0)))
    res = [None] * 8

    def work(i):
        res[i] = idx.knn_batch(q[i:i + 1], k)

    th = [threading.Thread(target=work, args=(i,)) for i in range(8)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    for i in range(8):
        _same(res[i], serial[i])
    b1, s1 = C.c_uint64(), C.c_uint64()
    V._lib.check(lib.vdb_batch_stats(idx.vec_set._h, C.byref(b1), C.byref(s1)))
    assert s1.value == s0.value, "large-k single-query calls must not go through the batcher"
    # vdb_parallel_knn: one vdb_flat_knn(nq = 1) per query from native threads
    ids = np.zeros((8, k), np.uint64)
    dd = np.zeros((8, k), np.float32)
    cnt = np.zeros(8, np.uint32)
    V._lib.check(lib.vdb_parallel_knn(idx.vec_set._h, V._lib.ptr(q), 8, k, 4, V._lib.ptr(ids), V._lib.ptr(dd),
                                      V._lib.ptr(cnt), None))
    _same((ids, dd, cnt), tuple(np.concatenate([s[j] for s in serial]) for j in range(3)))


def test_batch_spanning_several_chunks(vdb):
    """1400 queries over 200 000 rows: the emitted keys (8 bytes per row and query) take three 1 GiB chunks."""
    V = vdb
    V.init_devices([])
    n, nq, dim = 200_000, 1400, 16
    base, q = _data(n, nq, dim, 3, np.float32)
    idx = V.FlatIndex.from_vec_set(base, "l2sqr")
    kf = k_fused(dim, np.float32, nq)
    fused = idx.knn_batch(q, kf)
    got = idx.knn_batch(q, kf + 1)
    _same(got, fused, kf)
    assert (got[2] == kf + 1).all()
    _check_structure((got[0][::97], got[1][::97], got[2][::97]), n, kf + 1)


def test_ties_fall_to_the_lower_id(vdb):
    V = vdb
    V.init_devices([])
    dim = 32
    kf = k_fused(dim, np.float32, 1)
    # all rows identical: ids 0..k-1
    rows = np.tile(np.linspace(0, 1, dim, dtype=np.float32), (60_000, 1))
    q = np.full((1, dim), 0.25, np.float32)
    idx = V.FlatIndex.from_vec_set(rows, "l2sqr")
    ids, dd, cnt = idx.knn_batch(q, kf + 1)
    assert (ids[0].astype(np.int64) == np.arange(kf + 1)).all() and (dd[0] == dd[0, 0]).all()
    # two duplicate blocks at distance 0 that straddle rank k, in different shards of a 3-way split
    base, qq = _data(60_000, 1, dim, 4, np.float32)
    m = 12_000
    base[1_000:1_000 + m] = qq[0]
    base[45_000:45_000 + m] = qq[0]
    k = m + 4_000
    want_ids = np.concatenate([np.arange(1_000, 1_000 + m), np.arange(45_000, 45_000 + k - m)])
    full = V.FlatIndex.from_vec_set(base, "l2sqr")
    want = full.knn_batch(qq, k)
    assert (want[0][0].astype(np.int64) == want_ids).all() and (want[1][0] == 0).all()
    for devs in _device_sets():
        V.init_devices(devs)
        sidx = V.FlatIndex.from_vec_set(base, "l2sqr")
        _same(sidx.knn_batch(qq, k), want)
        del sidx
        V.init_devices([])


def test_small_sets(vdb):
    V = vdb
    V.init_devices([])
    base, q = _data(100, 3, 24, 5, np.float32)
    idx = V.FlatIndex.from_vec_set(base, "cosine")
    got = idx.knn_batch(q, 30_000)
    _check_structure(got, 100, 30_000)
    _same(got, idx.knn_batch(q, 100), 100)
    pairs = idx.knn(q[0], 30_000)                     # the trait's single-query call
    assert len(pairs) == 100


def _torch_ptr(t):
    return C.c_void_p(t.data_ptr())


def test_device_entry_points_and_key_merges(vdb):
    import torch
    V = vdb
    V.init_devices([])
    lib, L = V.lib(), V._lib
    n, nq, dim, k = 90_000, 5, 48, 40_000
    base, q = _data(n, nq, dim, 6, np.float32)
    idx = V.FlatIndex.from_vec_set(base, "l2sqr")
    want = idx.knn_batch(q, k)
    qd = torch.from_numpy(q).cuda()
    ids = torch.zeros((nq, k), dtype=torch.int64, device="cuda")
    dd = torch.zeros((nq, k), dtype=torch.float32, device="cuda")
    cnt = torch.zeros((nq,), dtype=torch.int32, device="cuda")
    keys = torch.zeros((nq, k), dtype=torch.int64, device="cuda")
    h = idx.vec_set._h
    L.check(lib.vdb_flat_knn_dev(h, _torch_ptr(qd), nq, k, _torch_ptr(ids), _torch_ptr(dd), _torch_ptr(cnt), None))
    torch.cuda.synchronize()
    _same((ids.cpu().numpy(), dd.cpu().numpy(), cnt.cpu().numpy()), want)
    for fn in (lib.vdb_flat_knn_keys_dev, lib.vdb_flat_scan_keys_dev):
        keys.zero_()
        L.check(fn(h, _torch_ptr(qd), nq, k, _torch_ptr(keys), None))
        L.check(lib.vdb_decode_keys_dev(_torch_ptr(keys), nq, k, _torch_ptr(ids), _torch_ptr(dd), _torch_ptr(cnt), None))
        torch.cuda.synchronize()
        _same((ids.cpu().numpy(), dd.cpu().numpy(), cnt.cpu().numpy()), want)
    # ascending padded lists of three row blocks (ids offset by id_base), merged: the unsharded result
    bounds = [(0, 20_000), (20_000, 55_000), (55_000, n)]
    lists = torch.zeros((3, nq, k), dtype=torch.int64, device="cuda")
    sets = []
    for s, (lo, hi) in enumerate(bounds):
        vs = V.DeviceVecSet(np.ascontiguousarray(base[lo:hi]), "l2sqr", id_base=lo)
        sets.append(vs)
        L.check(lib.vdb_flat_scan_keys_dev(vs._h, _torch_ptr(qd), nq, k, _torch_ptr(lists[s]), None))
    L.check(lib.vdb_merge_keys_dev(_torch_ptr(lists), 3, nq, k, _torch_ptr(ids), _torch_ptr(dd), _torch_ptr(cnt), None))
    torch.cuda.synchronize()
    _same((ids.cpu().numpy(), dd.cpu().numpy(), cnt.cpu().numpy()), want)
    merged = torch.zeros((nq, k), dtype=torch.int64, device="cuda")
    L.check(lib.vdb_merge_keys_to_keys_dev(_torch_ptr(lists), 3, nq, k, _torch_ptr(merged), None))
    L.check(lib.vdb_decode_keys_dev(_torch_ptr(merged), nq, k, _torch_ptr(ids), _torch_ptr(dd), _torch_ptr(cnt), None))
    torch.cuda.synchronize()
    _same((ids.cpu().numpy(), dd.cpu().numpy(), cnt.cpu().numpy()), want)
    # the tensor path keeps k <= 1024: forcing it with a larger k is still an error
    big, bq = _data(70_000, 4, 64, 7, np.float32)
    tidx = V.FlatIndex.from_vec_set(big, "l2sqr")
    tidx.vec_set.set_flat_path("tensor")
    with pytest.raises(Exception):
        tidx.knn_batch(bq, 2_000)


@pytest.mark.parametrize("metric,dtype", [("l2sqr", np.float32), ("cosine", np.uint8)])
def test_row_sharded_sets_equal_the_unsharded_call(vdb, metric, dtype):
    import torch
    V = vdb
    n, nq, dim = 60_000, 5, 64
    base, q = _data(n, nq, dim, 8, dtype)
    base[50_000] = base[3]            # an exact duplicate in another shard: the lower id first
    V.init_devices([])
    full = V.FlatIndex.from_vec_set(base, metric)
    ks = (k_fused(dim, dtype, nq) + 1, 30_000, n + 7)   # 30 000 and n + 7: larger than every shard
    want = {k: full.knn_batch(q, k) for k in ks}
    for devs in _device_sets():
        V.init_devices(devs)
        idx = V.FlatIndex.from_vec_set(base, metric)
        for k in ks:
            _same(idx.knn_batch(q, k), want[k])
        # device-resident call on adopted uneven shards
        g = len(devs)
        counts = [15_000] + [(n - 15_000) // (g - 1)] * (g - 1)
        counts[-1] += n - sum(counts)
        blocks, at = [], 0
        for s, d in enumerate(devs):
            blocks.append(torch.from_numpy(np.ascontiguousarray(base[at:at + counts[s]])).to(f"cuda:{d}"))
            at += counts[s]
        pitch = dim
        vs = V.DeviceVecSet.from_device_shards([b.data_ptr() for b in blocks], counts, devs, dim, pitch, dtype,
                                               metric, keepalive=blocks)
        didx = V.FlatIndex(vs)
        per = -(-nq // g)
        qd = [torch.from_numpy(q).to(f"cuda:{d}") for d in devs]
        for k in (ks[0], n + 7):
            ids = [torch.full((per, k), -1, dtype=torch.int64, device=f"cuda:{d}") for d in devs]
            dd = [torch.zeros((per, k), dtype=torch.float32, device=f"cuda:{d}") for d in devs]
            cnt = [torch.zeros((per,), dtype=torch.int32, device=f"cuda:{d}") for d in devs]
            didx.knn_batch_sharded_dev([t.data_ptr() for t in qd], nq, k, [t.data_ptr() for t in ids],
                                       [t.data_ptr() for t in dd], [t.data_ptr() for t in cnt])
            got = (torch.cat([t.cpu() for t in ids])[:nq].numpy(), torch.cat([t.cpu() for t in dd])[:nq].numpy(),
                   torch.cat([t.cpu() for t in cnt])[:nq].numpy())
            _same(got, want[k])
        del idx, didx, vs
        V.init_devices([])


def test_vecdb_search_with_k_len_and_upper_bound(vdb):
    V = vdb
    V.init_devices([])
    n, dim = 40_000, 32
    rows, q = _data(n, 1, dim, 9, np.float32)
    from lab_1806_vec_db_b200.table import VecDB
    db = VecDB()
    db.create_table_if_not_exists("t", dim)          # cosine, as the reference's default
    db.batch_add("t", rows.tolist(), [{"i": str(i)} for i in range(n)])
    full = V.FlatIndex.from_vec_set(rows, "cosine")
    ids, dist, cnt = full.knn_batch(q, n)
    r = float(dist[0, n // 2])                       # about 20 000 rows within r: more than the fused top-k holds
    got = db.search("t", q[0], k=len(db.tables["t"]), upper_bound=r)
    keep = dist[0] <= r
    assert len(got) == int(keep.sum()) > 16_000
    assert [m["i"] for m, _ in got] == [str(int(i)) for i in ids[0][keep]]
    assert np.array([d for _, d in got], np.float32).view(np.uint32).tolist() == dist[0][keep].view(np.uint32).tolist()
