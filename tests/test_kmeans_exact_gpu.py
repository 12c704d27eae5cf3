"""The index-building path of k-means bit for bit against the CPU oracle, at the shapes an index build runs.

Every centroid, codebook, weight, assignment and code here must equal the reference's sequential f32 arithmetic
(DESIGN.md section 2), so every comparison is on bits. Covered: the k-means++ weight update (k_means.rs:75-77), the
uniform-driven k-means++ pick rule (k_means.rs:61-87, `vdb_kmeans_pp_init_ds`), the batched PQ trainer's own k-means++
against the per-group path, Lloyd (k_means.rs:108-161) at IVF sizes, the assignment kernel's large-d shapes and its
dimension limit, and whole IVF / PQ builds under the reference's random stream (`rand_compat.StdRng`)."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

NTHREADS = os.cpu_count() or 1


@pytest.fixture(scope="module")
def V():
    import lab_1806_vec_db_b200 as V
    return V


def raw(a):
    """The bytes of an array: f32 bits or u8 values, compared exactly."""
    return np.ascontiguousarray(a).reshape(-1).view(np.uint8)


def gpu_pp_weights(rows, c, metric, w, sel):
    """`vdb_kmeans_pp_weights`: w[i] = min(w[i], d(c, rows[i][lo:hi])), w updated in place."""
    from lab_1806_vec_db_b200 import _lib as L
    rows, c = np.ascontiguousarray(rows), np.ascontiguousarray(c)
    n, dim = rows.shape
    L.check(L.lib().vdb_kmeans_pp_weights(L.ptr(rows), n, dim, L.dtype_code(rows), L.metric_code(metric), L.ptr(c),
                                          sel[0], sel[1], L.ptr(w)))
    return w


def pp_init_restated(oracle, rows, k, metric, sel, u):
    """The pick rule of `vdb_kmeans_pp_init_ds` on the oracle's weights: first pick floor(u0 n); per round r a sequential
    double total, target u[2r-1] * total and the first row whose running double sum exceeds it; the eagerly drawn
    fallback floor(u[2r] n) when a weight is negative, NaN or inf or the total is 0. Returns the chosen row indices."""
    n = rows.shape[0]
    lo, hi = sel

    def pick(x):
        return int(min(n - 1, np.floor(x * n)))

    chosen = [pick(u[0])]
    w = np.full(n, np.inf, np.float32)
    for r in range(1, k):
        w = oracle.kmeans_pp_weights(rows, rows[chosen[-1], lo:hi], metric, w, sel=sel, nthreads=NTHREADS)
        acc = np.cumsum(w.astype(np.float64))          # sequential, left to right
        nxt = pick(u[2 * r])
        if bool(np.all(w >= 0)) and not bool(np.isinf(w).any()) and acc[-1] > 0.0:
            target = u[2 * r - 1] * acc[-1]
            nxt = min(int(np.searchsorted(acc, target, side="right")), n - 1)
        chosen.append(nxt)
    return chosen


# ---- 2a: the k-means++ weight update ------------------------------------------------------------------------------------
def _pp_rows(rng, n, width, dtype):
    if dtype == "f32":
        rows = rng.standard_normal((n, width)).astype(np.float32)
    else:
        rows = rng.integers(0, 256, (n, width), dtype=np.uint8)
    if n > 2:
        rows[1] = rows[0]            # equal to the first round's centroid: weight 0
        rows[2] = 0                  # all-zero row: cosine's 1e-10 clamp
    return rows


@pytest.mark.parametrize("d", [1, 7, 31, 32, 33, 40, 129, 960, 1500])
@pytest.mark.parametrize("metric", ["l2sqr", "cosine"])
@pytest.mark.parametrize("dtype", ["f32", "u8"])
def test_pp_weights_bit_exact(V, oracle, d, metric, dtype):
    """Two rounds and more of the update, the first from +inf, the next from the previous output (so `min` keeps old
    weights for part of the rows), on the full row and on a window with lo > 0; the last round's centroid is the
    all-zero row."""
    rng = np.random.default_rng(1000 * d + (metric == "cosine") * 10 + (dtype == "u8"))
    for n in (1, 37, 5000):
        wide = _pp_rows(rng, n, d + 5, dtype)
        for rows, sel in ((np.ascontiguousarray(wide[:, 3:3 + d]), (0, d)), (wide, (3, 3 + d))):
            lo, hi = sel
            w_gpu = np.full(n, np.inf, np.float32)
            w_orc = w_gpu.copy()
            for c in dict.fromkeys((0, n // 2, min(2, n - 1))):
                cen = np.ascontiguousarray(rows[c, lo:hi])
                gpu_pp_weights(rows, cen, metric, w_gpu, sel)
                w_orc = oracle.kmeans_pp_weights(rows, cen, metric, w_orc, sel=sel, nthreads=NTHREADS)
                bad = np.nonzero(raw(w_gpu).view(np.uint32) != raw(w_orc).view(np.uint32))[0]
                assert bad.size == 0, (f"n={n} sel={sel} centroid row {c}: {bad.size} weights differ in bits, e.g. row "
                                       f"{bad[0]}: {w_gpu[bad[0]]!r} vs {w_orc[bad[0]]!r}")
            if metric == "l2sqr":
                assert w_gpu[0] == 0.0
            if n > 2:
                assert w_gpu[2] == (0.0 if metric == "l2sqr" else 1.0)


@pytest.mark.parametrize("metric", ["l2sqr", "cosine"])
def test_pp_weights_u8_sums_beyond_2_pow_24(V, oracle, metric):
    """u8 rows of bytes 180-255 against a centroid of bytes 0-40 at d = 960: the squared sums pass 2^24, where the
    sequential f32 chain rounds. k-means parity is that rounded value (no integer exception as in Flat's u8 path)."""
    rng = np.random.default_rng(24)
    rows = rng.integers(180, 256, (3000, 960), dtype=np.uint8)
    rows[7] = rng.integers(0, 41, 960, dtype=np.uint8)
    c = np.ascontiguousarray(rows[7])
    exact = ((rows.astype(np.int64) - c.astype(np.int64)) ** 2).sum(1)
    assert (exact > (1 << 24)).sum() > 2900
    w = gpu_pp_weights(rows, c, metric, np.full(3000, np.inf, np.float32), (0, 960))
    want = oracle.kmeans_pp_weights(rows, c, metric, np.full(3000, np.inf, np.float32), nthreads=NTHREADS)
    assert (raw(w) == raw(want)).all()
    if metric == "l2sqr":   # the rounded chain is not the integer: the parity target really is the rounded value
        assert (want.astype(np.float64) != exact.astype(np.float64)).any()


# ---- 2c: uniform-driven k-means++ (vdb_kmeans_pp_init_ds) ------------------------------------------------------------------
@pytest.mark.parametrize("case", ["f32_l2sqr", "f32_cosine_window", "u8_l2sqr", "k1", "k_gt_n", "identical_window"])
def test_pp_init_bit_exact_vs_restated_pick_rule(V, oracle, case):
    rng = np.random.default_rng(sum(map(ord, case)))
    metric, k, sel, dtype, n, dim = "l2sqr", 24, None, "f32", 5000, 960
    if case == "f32_cosine_window":
        metric, sel, dim = "cosine", (30, 330), 400
    elif case == "u8_l2sqr":
        dtype, dim = "u8", 128
    elif case == "k1":
        k = 1
    elif case == "k_gt_n":
        n, dim, k = 20, 17, 30
    elif case == "identical_window":
        n, dim, sel = 800, 64, (10, 40)
    rows = (rng.standard_normal((n, dim)).astype(np.float32) if dtype == "f32"
            else rng.integers(0, 256, (n, dim), dtype=np.uint8))
    if case == "identical_window":
        rows[:, 10:40] = rows[3, 10:40]          # every weight 0 after the first round: every pick is the fallback
    sel = sel if sel is not None else (0, dim)
    seed = 77 + k
    u = np.random.default_rng(seed).random(2 * k - 1)
    got = V.k_means_init(rows, V.KMeansConfig(k, 5, 1e-6, metric, sel), np.random.default_rng(seed))
    chosen = pp_init_restated(oracle, rows, k, metric, sel, u)
    want = np.ascontiguousarray(rows[chosen, sel[0]:sel[1]])
    assert got.shape == want.shape and (raw(got) == raw(want)).all(), chosen
    if case == "k_gt_n":
        assert len(set(chosen)) == n           # every row is taken before the fallback starts repeating them
    if case == "identical_window":
        assert chosen[1:] == [int(min(n - 1, np.floor(u[2 * r] * n))) for r in range(1, k)]


# ---- 2d: the batched PQ trainer without initial codebooks vs the per-group path --------------------------------------------
@pytest.mark.parametrize("n_bits", [4, 8])
@pytest.mark.parametrize("metric", ["l2sqr", "cosine"])
@pytest.mark.parametrize("dtype", ["f32", "u8"])
def test_batched_pq_training_from_uniforms_vs_per_group(V, n_bits, metric, dtype):
    """train_codebooks (one launch of pq_train_kernel: k-means++ from m x (2k-1) uniforms, then Lloyd) against
    KMeans.from_vec_set per group on the same Generator (vdb_kmeans_pp_init_ds + vdb_kmeans_train_ds). n = 10 000 rows
    puts about 40 rows in each thread's chunk, so picks land in late chunks; one group's sub-vectors are all identical."""
    from lab_1806_vec_db_b200.index import train_codebooks
    n, dim, m, iters = 10_000, 43, 9, 8
    k = 1 << n_bits
    # both paths draw m x (2k - 1) uniforms in group order from the same stream
    a = np.random.default_rng(3).random((m, 2 * k - 1))
    g = np.random.default_rng(3)
    assert (a == np.stack([g.random(2 * k - 1) for _ in range(m)])).all()
    rng = np.random.default_rng(10 * n_bits + (metric == "cosine") * 2 + (dtype == "u8"))
    rows = (rng.random((n, dim), dtype=np.float32) if dtype == "f32"
            else rng.integers(0, 256, (n, dim), dtype=np.uint8))
    groups = V.pq_groups(dim, m)
    lo, hi = groups[2]
    rows[:, lo:hi] = rows[5, lo:hi]
    vs = V.DeviceVecSet(rows, metric)
    cfg = V.PQConfig(n_bits, m, metric, None, iters, 1e-6)
    books = train_codebooks(vs, cfg, np.random.default_rng(3))
    got_iters = train_codebooks.last_iterations.copy()
    g = np.random.default_rng(3)
    parts, want_iters = [], []
    for lo, hi in groups:
        km = V.KMeans.from_vec_set(vs, V.KMeansConfig(k, iters, 1e-6, metric, (lo, hi)), g)
        parts.append(km.centroids.reshape(-1))
        want_iters.append(km.iterations)
    want = np.concatenate(parts)
    off = np.cumsum([0] + [k * (hi - lo) for lo, hi in groups])
    bad = [gi for gi in range(m) if (raw(books[off[gi]:off[gi + 1]]) != raw(want[off[gi]:off[gi + 1]])).any()]
    assert not bad, f"codebooks of groups {bad} differ"
    assert got_iters.tolist() == want_iters
    assert want_iters[2] == 1                  # identical sub-vectors converge at once


# ---- 2e: Lloyd at build sizes ----------------------------------------------------------------------------------------------
def _lloyd_case(rng, case):
    """(rows, init centroids, metric, sel, max_iter)"""
    if case == "ivf_100k_960_k128":
        rows = rng.random((100_000, 960), dtype=np.float32)
        return rows, rows[rng.choice(len(rows), 128, replace=False)], "l2sqr", None, 8
    if case == "cosine_50k_300_k100":
        rows = rng.standard_normal((50_000, 300)).astype(np.float32)
        return rows, rows[rng.choice(len(rows), 100, replace=False)], "cosine", None, 5
    if case == "u8_128_k64":
        rows = rng.integers(0, 256, (20_000, 128), dtype=np.uint8)
        rows[:, :8] = 255                         # means of exactly 255: the saturating edge of `as u8`
        rows[:, 8:16] = rng.integers(254, 256, (20_000, 8), dtype=np.uint8)   # means in (254, 255): truncate to 254
        rows[:, 16:20] = 0
        return rows, rows[rng.choice(len(rows), 64, replace=False)], "l2sqr", None, 6
    if case == "f32_window_duplicates":
        rows = rng.random((30_000, 301), dtype=np.float32)
        init = np.ascontiguousarray(rows[rng.choice(len(rows), 40, replace=False), 5:290])
        init[5] = init[17] = 10.0                 # two equal centroids far from every row: both clusters stay empty
        return rows, init, "l2sqr", (5, 290), 6
    raise AssertionError(case)


@pytest.mark.parametrize("case", ["ivf_100k_960_k128", "cosine_50k_300_k100", "u8_128_k64", "f32_window_duplicates"])
def test_lloyd_bit_exact_at_build_sizes(V, oracle, case):
    """Lloyd from the same initial centroids: centroid bits and iteration count. The IVF shape (100 000 x 960, k = 128)
    runs the update with more than one dimension per thread (d > 256), clusters of thousands of members, the assignment
    grid with several row-steps per warp and the best key carried across four centroid chunks."""
    rows, init, metric, sel, max_iter = _lloyd_case(np.random.default_rng(len(case)), case)
    init = np.ascontiguousarray(init)
    want, it_want = oracle.kmeans_lloyd(rows, init, metric, max_iter, 1e-6, sel=sel)
    km = V.KMeans.from_vec_set(rows, V.KMeansConfig(init.shape[0], max_iter, 1e-6, metric, sel), init_centroids=init)
    assert km.iterations == it_want
    diff = np.nonzero((km.centroids != want).any(1) if rows.dtype == np.uint8 else
                      (km.centroids.view(np.uint32) != want.view(np.uint32)).any(1))[0]
    assert diff.size == 0, f"centroids {diff[:10]} differ"
    if case == "f32_window_duplicates":   # the empty clusters kept their centroid
        assert (raw(km.centroids[5]) == raw(init[5])).all() and (raw(km.centroids[17]) == raw(init[17])).all()
    if case == "u8_128_k64":
        assert (km.centroids[:, :8] == 255).all() and (km.centroids[:, 16:20] == 0).all()
        assert (km.centroids[:, 8:16] == 254).any()


# ---- 2f: large-d assignment and the dimension limit ------------------------------------------------------------------------
@pytest.mark.parametrize("d", [2048, 4096, 5685])
@pytest.mark.parametrize("k", [1, 3, 40])
def test_assign_large_d(V, oracle, d, k):
    """d between 1500 and 5685 makes the assignment kernel fall back to one row per warp step and narrow centroid
    chunks (d = 5685: one centroid and one row, the last shape that fits its shared memory)."""
    rng = np.random.default_rng(d + k)
    rows = rng.random((1500, d), dtype=np.float32)
    cent = np.ascontiguousarray(rows[rng.choice(len(rows), k, replace=False)] + np.float32(0.01))
    if k > 2:
        cent[k - 1] = cent[1]                     # exact duplicate: ties go to the lower id
    want = oracle.kmeans_assign(rows, cent, "l2sqr", nthreads=NTHREADS)
    km = V.KMeans(V.KMeansConfig(k, dist="l2sqr"), cent)
    assert (km.find_nearest_batch(rows) == want).all()
    vs = V.DeviceVecSet(rows, "l2sqr")
    ivf = V.IVFIndex(vs, cent)
    assert (ivf.assignment == want).all()
    if k == 40:
        assert len(np.unique(want)) > 20


def test_assign_refuses_d_5686(V):
    """One dimension more than fits: a clean error from both entry points, not a result."""
    rows = np.random.default_rng(1).random((64, 5686), dtype=np.float32)
    km = V.KMeans(V.KMeansConfig(2, dist="l2sqr"), rows[:2])
    with pytest.raises(V.VdbError, match="too large"):
        km.find_nearest_batch(rows)
    vs = V.DeviceVecSet(rows, "l2sqr")
    with pytest.raises(V.VdbError, match="too large"):
        V.IVFIndex(vs, rows[:2])


# ---- 2g: whole builds under the reference's random stream -------------------------------------------------------------------
def test_ivf_build_under_reference_stream(V, oracle):
    """IVFIndex.from_vec_set with StdRng: sample = shuffle(n)[:size], k-means++ picks from the oracle's weights, Lloyd
    and the list assignment of every row - all bit for bit."""
    from lab_1806_vec_db_b200.rand_compat import StdRng, k_means_init_indices
    rng = np.random.default_rng(64)
    rows = rng.random((30_000, 128), dtype=np.float32)
    cfg = V.IVFConfig(64, 20_000, 5, 1e-6)
    vs = V.DeviceVecSet(rows, "l2sqr")
    ivf = V.IVFIndex.from_vec_set(vs, rows, "l2sqr", cfg, StdRng.seed_from_u64(7))

    s = StdRng.seed_from_u64(7)
    train = np.ascontiguousarray(rows[s.shuffle(len(rows))[:cfg.k_means_size]])
    w = [np.full(len(train), np.inf, np.float32)]

    def update(idx):
        w[0] = oracle.kmeans_pp_weights(train, train[idx], "l2sqr", w[0], nthreads=NTHREADS)
        return w[0]

    picks = k_means_init_indices(update, len(train), cfg.k, s)
    cent, _ = oracle.kmeans_lloyd(train, train[picks], "l2sqr", cfg.k_means_max_iter, cfg.k_means_tol)
    assert (raw(ivf.centroids) == raw(cent)).all()
    assert (ivf.assignment == oracle.kmeans_assign(rows, cent, "l2sqr", nthreads=NTHREADS)).all()


@pytest.mark.parametrize("metric", ["l2sqr", "cosine"])
def test_pq_build_under_reference_stream(V, oracle, metric):
    """PQTable.from_vec_set with StdRng: the sample, each group's k-means++ in group order on one stream, Lloyd per group
    and the codes of every row - all bit for bit."""
    from lab_1806_vec_db_b200.rand_compat import StdRng, k_means_init_indices
    rng = np.random.default_rng(16)
    rows = rng.random((12_000, 100), dtype=np.float32)
    cfg = V.PQConfig(4, 16, metric, 5000, 5, 1e-6)
    vs = V.DeviceVecSet(rows, metric)
    pq = V.PQTable.from_vec_set(vs, rows, cfg, StdRng.seed_from_u64(11))

    s = StdRng.seed_from_u64(11)
    train = np.ascontiguousarray(rows[s.shuffle(len(rows))[:cfg.k_means_size]])
    books = []
    for lo, hi in oracle.pq_groups(rows.shape[1], cfg.m):
        w = [np.full(len(train), np.inf, np.float32)]

        def update(idx):
            w[0] = oracle.kmeans_pp_weights(train, train[idx, lo:hi], metric, w[0], sel=(lo, hi), nthreads=NTHREADS)
            return w[0]

        picks = k_means_init_indices(update, len(train), 16, s)
        cb, _ = oracle.kmeans_lloyd(train, train[picks, lo:hi], metric, cfg.k_means_max_iter, cfg.k_means_tol,
                                    sel=(lo, hi))
        books.append(cb.reshape(-1))
    books = np.concatenate(books)
    assert (raw(pq.codebooks) == raw(books)).all()
    codes = oracle.pq_encode(rows, books, cfg.m, cfg.n_bits, metric, nthreads=NTHREADS)
    assert (pq.encoded_vec_set == codes).all()
