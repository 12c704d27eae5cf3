"""HNSW on data where every distance is exact: the oracle's batched build, its tie-event counts and the bound that
makes a dot product exact in any summation order. tests/test_hnsw_exact_gpu.py compares the device kernels with these
restatements bit for bit; the helpers below are shared with it.

Integer-valued rows, queries and codebooks with every partial sum below 2^24 make each dot product, squared norm,
lookup-table entry and ADC sum an exact f32 integer whatever the order of the additions. The remaining operations of a
distance (one add or product, sqrt, max, one division) are single IEEE operations on identical inputs on both sides, so
the device and the oracle compute the same bits. Two correct walks over the same graph then differ only where the
oracle meets an exact distance tie on a full result set (a "tie event")."""
import numpy as np
import pytest

EXACT_LIMIT = 2 ** 24


def exact_rows(rng, n, dim, dtype, lo, hi):
    """n integer-valued rows in [lo, hi] of `dtype`"""
    return rng.integers(lo, hi + 1, (n, dim)).astype(dtype)


def assert_exact(*arrays, pq_l2=False):
    """The data of a test is exact: integer values, and 2 * dim * R^2 < 2^24 with R the largest magnitude (a squared
    norm, a dot product and their sum in the cached L2 form stay below 2^24). With pq_l2 the L2 lookup entries are sums
    of (q - c)^2, and their ADC sum over all groups must stay below 2^24 too: dim * (2R)^2 for signed values, dim * R^2
    for unsigned ones."""
    dim = arrays[0].shape[-1]
    r, signed = 0, False
    for a in arrays:
        if a.size == 0:
            continue
        v = np.asarray(a, np.float64)
        assert (v == np.round(v)).all(), "test data must be integer-valued"
        r = max(r, int(np.abs(v).max()))
        signed = signed or bool((v < 0).any())
    bound = 2 * dim * r * r
    if pq_l2:
        bound = max(bound, dim * (2 * r if signed else r) ** 2)
    assert bound < EXACT_LIMIT, f"dim {dim}, R {r}: partial sums up to {bound} are not exact in f32"
    return bound


def differing_lists(a, b):
    """The number of adjacency lists (level 0 and upper levels) in which two graphs differ. a, b: (links0 [n, 2M],
    len0 [n], ulinks [slots * M], ulen [slots]) in the layouts of HNSWIndex.level0_links / upper_links."""
    l0a, n0a, ula, una = a
    l0b, n0b, ulb, unb = b
    m = l0a.shape[1] // 2
    bad = sum(int(n0a[i] != n0b[i] or (l0a[i, :n0a[i]] != l0b[i, :n0b[i]]).any()) for i in range(len(n0a)))
    bad += sum(int(una[s] != unb[s] or (ula[s * m:s * m + una[s]] != ulb[s * m:s * m + unb[s]]).any())
               for s in range(len(una)))
    return bad


def oracle_graph(h):
    return (*h.links0(), *h.upper())


def same_graph(a, b):
    return differing_lists(oracle_graph(a), oracle_graph(b))


@pytest.mark.parametrize("dtype,metric,dim,lo,hi,M", [
    (np.float32, "l2sqr", 64, -300, 300, 8),
    (np.uint8, "cosine", 17, 0, 255, 2),
    (np.float32, "cosine", 3, -1000, 1000, 4),
    (np.uint8, "l2sqr", 100, 0, 255, 32),
])
def test_batched_build_with_batches_of_one_is_the_sequential_build(oracle, dtype, metric, dim, lo, hi, M):
    """orc_hnsw_build_batched(max_batch = 1) inserts one node per batch, searching the graph as it stood before it:
    that is the reference's `add`, so the graph, the enter point and the tie count equal orc_hnsw_build's."""
    from oracle.oracle_py import HnswOracle
    from lab_1806_vec_db_b200.index import hnsw_rand_levels
    rng = np.random.default_rng(dim * 100 + M)
    n = 1500
    base = exact_rows(rng, n, dim, dtype, lo, hi)
    assert_exact(base)
    levels = hnsw_rand_levels(n, M, rng)
    seq = HnswOracle(base, metric, M, 60, levels)
    one = HnswOracle.batched(base, metric, M, 60, levels, max_batch=1)
    assert same_graph(seq, one) == 0
    assert one.enter_point == (int(np.argmax(levels == levels.max())), int(levels.max()))
    assert seq.build_ties == one.build_ties
    # build + append with batches of one is the same sequence of inserts
    app = HnswOracle.batched(base, metric, M, 60, levels, max_batch=1, n0=n // 3)
    assert same_graph(seq, app) == 0 and app.enter_point == one.enter_point


def test_batched_build_searches_the_graph_as_the_batch_found_it(oracle):
    """With batches larger than one the new nodes of a batch do not see each other's links, only the brute-force
    candidates among the batch: a different graph from the sequential one, but a valid one (no self links, no
    duplicates, lists within M / 2M), and an append's batches start over at the rows it adds."""
    from oracle.oracle_py import HnswOracle
    from lab_1806_vec_db_b200.index import hnsw_rand_levels
    rng = np.random.default_rng(7)
    n, dim, M = 3000, 24, 4
    base = exact_rows(rng, n, dim, np.float32, -300, 300)
    assert_exact(base)
    levels = hnsw_rand_levels(n, M, rng)
    seq = HnswOracle(base, "l2sqr", M, 40, levels)
    bat = HnswOracle.batched(base, "l2sqr", M, 40, levels, max_batch=64)
    assert same_graph(seq, bat) > 0          # batches of up to 64 nodes really were formed
    links, lens = bat.links0()
    assert lens.max() <= 2 * M and (lens[1:] > 0).all()
    for i in range(n):
        row = links[i, :lens[i]]
        assert (row < n).all() and (row != i).all() and len(set(row.tolist())) == len(row)
    ul, un = bat.upper()
    assert un.size == 0 or un.max() <= M
    # recall of the batched graph is as good as the sequential one's on this easy set
    q = exact_rows(rng, 100, dim, np.float32, -300, 300)
    gt = oracle.flat_knn(base, q, 10, "l2sqr", nthreads=oracle.ncores())[0]
    r = [np.mean([len(set(a) & set(b)) / 10 for a, b in zip(h.knn(q, 10, 80, nthreads=4)[0].tolist(), gt.tolist())])
         for h in (seq, bat)]
    assert r[1] >= r[0] - 0.02, r
    # an append restarts the batch sizes at done = n0: batches cut at row 1000, so not the one-shot build's graph
    app = HnswOracle.batched(base, "l2sqr", M, 40, levels, max_batch=64, n0=1000)
    assert same_graph(bat, app) > 0


def test_duplicate_rows_are_counted_as_tie_events(oracle):
    """A row repeated many times gives equal distances on a full result set: the build and a search on that row count
    them; a query whose nearest row is unique, with a result set of one, counts none."""
    from oracle.oracle_py import HnswOracle
    rng = np.random.default_rng(3)
    dim, M = 8, 4
    base = exact_rows(rng, 200, dim, np.float32, -50, 50)
    base[:30] = base[0]                                  # 30 copies of one row
    assert_exact(base)
    levels = np.zeros(200, np.uint32)
    h = HnswOracle(base, "l2sqr", M, 2 * M, levels)      # 9 copies reachable from row 0, a candidate set of 8
    assert h.build_ties > 0
    ids, dd, cnt, ties = h.knn(base[:1], 3, 3, ties=True)
    assert ties[0] > 0 and cnt[0] == 3 and (dd[0] == 0).all() and (ids[0] < 30).all()
    assert HnswOracle.batched(base, "l2sqr", M, 2 * M, levels, max_batch=8).build_ties > 0
    # a row far from the rest, searched with ef = 1: the set of one never meets an equal distance
    solo = np.concatenate([base, np.full((1, dim), 1000, np.float32)])
    h2 = HnswOracle(solo, "l2sqr", M, 10, np.zeros(201, np.uint32))
    *_, t2 = h2.knn(solo[200:], 1, 1, ties=True)
    assert t2.tolist() == [0]


def test_pq_resort_ties_are_counted(oracle):
    """knn_pq's tie count adds the resort's: two identical rows with equal exact distances on a k = 1 resort."""
    from oracle.oracle_py import HnswOracle
    rng = np.random.default_rng(5)
    base = exact_rows(rng, 300, 8, np.float32, -20, 20)
    base[1] = base[0]
    m = 4
    books = np.concatenate([base[10:26, lo:hi].reshape(-1) for lo, hi in oracle.pq_groups(8, m)])
    assert_exact(base, books, pq_l2=True)
    codes = oracle.pq_encode(base, books, m, 4, "l2sqr")
    h = HnswOracle(base, "l2sqr", 4, 40, np.zeros(300, np.uint32))
    ids, dd, cnt, ties = h.knn_pq(base[:1], 1, 300, codes, books, m, 4, ties=True)
    assert ids[0, 0] in (0, 1) and dd[0, 0] == 0 and ties[0] >= 1


def test_the_exactness_bound():
    """assert_exact accepts the largest R a dimension allows and rejects the next"""
    assert_exact(np.full((1, 1025), 90, np.float32))
    with pytest.raises(AssertionError):
        assert_exact(np.full((1, 1025), 91, np.float32))
    assert_exact(np.full((1, 2050), 63, np.uint8), pq_l2=True)
    with pytest.raises(AssertionError):
        assert_exact(np.array([[-200] * 64 + [100] * 64], np.float32), pq_l2=True)   # 128 * 400^2 >= 2^24
    with pytest.raises(AssertionError):
        assert_exact(np.array([[0.5, 1.0]], np.float32))
