"""`not gpu`: pins the CPU oracle against the reference's own known-answer tests and against the
golden vectors produced by the independent numpy emulation (tests/golden/make_golden.py)."""
import hashlib
import os

import numpy as np
import pytest


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def test_fixture_checksums(fixtures):
    """The re-encoded fixtures reproduce the reference's data files bit for bit."""
    assert hashlib.sha256(fixtures["base"].tobytes()).hexdigest() == fixtures["base_sha256"]
    assert hashlib.sha256(fixtures["test"].tobytes()).hexdigest() == fixtures["test_sha256"]
    assert fixtures["base_sha256"].startswith("b21021ce") and fixtures["test_sha256"].startswith("5779751c")
    assert (fixtures["base"][50] == fixtures["base"][444]).all()  # the known exact duplicate


def test_reference_distance_known_answers(oracle):
    """distance/mod.rs:138-150."""
    a, b = np.array([1, 2, 3], np.float32), np.array([4, 5, 6], np.float32)
    assert abs(oracle.distance(a, b, "l2sqr") - 27.0) < 1e-6
    a8, b8 = np.array([1, 2, 3], np.uint8), np.array([2, 4, 6], np.uint8)
    assert abs(oracle.distance(a8, b8, "cosine") - 0.0) < 1e-6


def test_reference_pq_groups_known_answers(oracle):
    """pq_table.rs:312-322."""
    assert oracle.pq_groups(6, 2) == [(0, 3), (3, 6)]
    assert oracle.pq_groups(7, 3) == [(0, 3), (3, 5), (5, 7)]
    assert oracle.pq_groups(960, 240) == [(4 * i, 4 * i + 4) for i in range(240)]
    with pytest.raises(AssertionError):
        oracle.pq_groups(3, 5)


@pytest.mark.parametrize("metric", ["l2sqr", "cosine"])
def test_flat_golden_sha_anchors(fixtures, golden, oracle, metric):
    """C1 (gist_1000 x gist_test, k=10): oracle == numpy emulation, bit for bit, and the SHA-256
    anchors of SURVEY.md section 8(c)."""
    ids, dd, cnt = oracle.flat_knn(fixtures["base"], fixtures["test"], 10, metric, os.cpu_count())
    assert (cnt == 10).all()
    assert (ids.astype(np.int64) == golden[f"flat_{metric}_ids"]).all()
    assert (bits(dd) == bits(golden[f"flat_{metric}_dist"])).all()
    anchors = {
        "l2sqr": ("f2ac163d5b4dd167f90259874b4c1325373358dfc500aedba14ff9a96860f844",
                  "416b9c67360cb8b64f1777cdeae9c297aaf4f6a90afb0ee93bf9b78484fbc222"),
        "cosine": ("689905afd78cfee1f0694fafd61508ff74434b53a138974846748363606bbc48",
                   "d51df5095c010ccd6c62d5a46f61e18e2c6e20b583c82611305b9208081e1073"),
    }[metric]
    assert hashlib.sha256(ids.astype("<i8").tobytes()).hexdigest() == anchors[0]
    assert hashlib.sha256(dd.astype("<f4").tobytes()).hexdigest() == anchors[1]
    if metric == "l2sqr":
        assert ids[0].tolist() == [918, 467, 725, 988, 207, 56, 18, 348, 27, 632]
        assert ids[19, :2].tolist() == [50, 444]


@pytest.mark.parametrize("metric", ["l2sqr", "cosine"])
def test_flat_unit_shape(fixtures, golden, oracle, metric):
    """flat_index.rs:117-170 shape: dim clipped to 12, query = row 200."""
    b12 = np.ascontiguousarray(fixtures["base"][:, :12])
    ids, dd, _ = oracle.flat_knn(b12, b12[200:201], 6, metric)
    assert (ids.astype(np.int64) == golden[f"unit12_{metric}_ids"]).all()
    assert (bits(dd) == bits(golden[f"unit12_{metric}_dist"])).all()
    assert ids[0, 0] == 200 and abs(dd[0, 0]) < 1e-6


@pytest.mark.parametrize("metric", ["l2sqr", "cosine"])
def test_assign_and_ivf_golden(fixtures, golden, oracle, metric):
    base, test = fixtures["base"], fixtures["test"]
    cent = np.ascontiguousarray(base[7:23])
    a = oracle.kmeans_assign(base, cent, metric)
    assert (a == golden[f"assign16_{metric}"]).all()
    off, mem = oracle.ivf_lists(a, 16)
    ids, dd, cnt = oracle.ivf_knn(base, cent, off, mem, test[:50], 10, 4, metric)
    assert (ids.astype(np.int64) == golden[f"ivf_{metric}_ids"]).all()
    assert (bits(dd) == bits(golden[f"ivf_{metric}_dist"])).all()


def test_assign_selected_range(fixtures, golden, oracle):
    base = fixtures["base"]
    cent = np.ascontiguousarray(base[7:23, 100:113])
    assert (oracle.kmeans_assign(base, cent, "l2sqr", sel=(100, 113)) == golden["assign16_sel_l2sqr"]).all()


@pytest.mark.parametrize("tag,m,n_bits,dimclip", [("pq240", 240, 4, 960), ("pq7", 7, 4, 13), ("pq5b8", 5, 8, 13)])
@pytest.mark.parametrize("metric", ["l2sqr", "cosine"])
def test_pq_golden(fixtures, golden, oracle, tag, m, n_bits, dimclip, metric):
    rows = np.ascontiguousarray(fixtures["base"][:200, :dimclip])
    cb = golden[f"{tag}_codebooks"]
    codes = oracle.pq_encode(rows, cb, m, n_bits, metric)
    assert (codes == golden[f"{tag}_{metric}_codes"]).all()
    dc = oracle.pq_dist_cache(dimclip, cb, m, n_bits, metric)
    assert (bits(dc) == bits(golden[f"{tag}_{metric}_dist_cache"])).all()
    for qi in range(5):
        q = np.ascontiguousarray(fixtures["test"][qi, :dimclip])
        lut, qc = oracle.pq_lookup(q, cb, m, n_bits, metric)
        assert (bits(lut) == bits(golden[f"{tag}_{metric}_lut"][qi])).all()
        assert np.float32(qc) == golden[f"{tag}_{metric}_qcache"][qi]
        adc = oracle.pq_adc(codes, m, n_bits, metric, lut, dc, qc)
        assert (bits(adc) == bits(golden[f"{tag}_{metric}_adc"][qi])).all()
    ids, dd, _ = oracle.flat_knn_pq(rows, codes, cb, m, n_bits, np.ascontiguousarray(fixtures["test"][:5, :dimclip]),
                                    10, 40, metric)
    assert (ids.astype(np.int64) == golden[f"{tag}_{metric}_knn_ids"]).all()
    assert (bits(dd) == bits(golden[f"{tag}_{metric}_knn_dist"])).all()


@pytest.mark.parametrize("metric", ["l2sqr", "cosine"])
def test_pq_precise_when_points_fewer_than_centroids(oracle, metric):
    """pq_table.rs:324-372: 5 vectors, m=2, 4 bits (16 centroids > 5 points) -> ADC == exact distance."""
    rng = np.random.default_rng(42)
    rows = rng.random((5, 8), dtype=np.float32)
    cbs = []
    for lo, hi in oracle.pq_groups(8, 2):
        c = np.zeros((16, hi - lo), np.float32)
        c[:5] = rows[:, lo:hi]
        c[5:] = 1e3 + np.arange(11)[:, None]  # far away, never chosen
        cbs.append(c.reshape(-1))
    cb = np.concatenate(cbs)
    codes = oracle.pq_encode(rows, cb, 2, 4, metric)
    dc = oracle.pq_dist_cache(8, cb, 2, 4, metric)
    for i in range(5):
        lut, qc = oracle.pq_lookup(rows[i], cb, 2, 4, metric)
        adc = oracle.pq_adc(codes, 2, 4, metric, lut, dc, qc)
        for j in range(5):
            assert abs(adc[j] - oracle.distance(rows[i], rows[j], metric)) < 1e-6


@pytest.mark.parametrize("metric", ["l2sqr", "cosine"])
def test_cached_forms_golden(fixtures, golden, oracle, metric):
    """hnsw_index.rs:351-358 / distance/mod.rs:54-57, 67-69."""
    base, q = fixtures["base"], fixtures["test"][3]
    cache = np.array([oracle.dist_cache(r, metric) for r in base], np.float32)
    assert (bits(cache) == bits(golden[f"cached_{metric}_rowcache"])).all()
    cand = np.arange(0, 1000, 7)
    d = oracle.gather_dist(base, cache, q, oracle.dist_cache(q, metric), cand, metric)
    assert (bits(d) == bits(golden[f"cached_{metric}_dist"])).all()


def test_kmeans_on_real_set_property(fixtures, oracle):
    """k_means.rs:241-277: k=3 on dims 0..5 of a 400-row sample; find_nearest(centroid[1]) == 1."""
    rows = np.ascontiguousarray(fixtures["base"][:400])
    init = oracle.kmeans_pp_init(rows, 3, "l2sqr", seed=42, sel=(0, 5))
    cent, iters = oracle.kmeans_lloyd(rows, init, "l2sqr", 20, 1e-6, sel=(0, 5))
    assert cent.shape == (3, 5) and 1 <= iters <= 20
    v = np.zeros(960, np.float32)
    v[:5] = cent[1]
    assert oracle.kmeans_assign(v.reshape(1, -1), cent, "l2sqr", sel=(0, 5))[0] == 1


@pytest.mark.parametrize("metric", ["l2sqr", "cosine"])
@pytest.mark.parametrize("dtype", ["f32", "u8"])
def test_kmeans_pp_weights_equals_numpy_emulation(fixtures, oracle, metric, dtype):
    """k_means.rs:75-77: w[i] = min(w[i], d(c, v_i)) on the whole row and on a window with lo > 0, two rounds (the second
    keeps the smaller old weight for part of the rows), split across threads: bit for bit the numpy emulation's
    sequential f32 distance. A row equal to the centroid gets weight 0."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import np_emul as E
    base = fixtures["base"][:300]
    rows = base if dtype == "f32" else np.clip(np.rint(base * 255.0), 0, 255).astype(np.uint8)
    for lo, hi in ((0, rows.shape[1]), (37, 170)):
        sub = rows[:, lo:hi]
        want = np.full(len(rows), np.inf, np.float32)
        got = want.copy()
        for c in (11, 250):
            d = E.distance(np.broadcast_to(sub[c], sub.shape), sub, metric)
            want = np.fmin(want, d).astype(np.float32)
            got = oracle.kmeans_pp_weights(rows, sub[c], metric, got, sel=(lo, hi), nthreads=4)
            assert (bits(got) == bits(want)).all(), (lo, hi, c)
            assert got[c] == 0.0 or metric == "cosine"
        kept = bits(got) != bits(E.distance(np.broadcast_to(sub[250], sub.shape), sub, metric))
        assert kept.any() and not kept.all()


def test_lloyd_empty_cluster_and_u8_cast(oracle):
    """k_means.rs:131-137 (empty cluster keeps its centroid) and scalar.rs:22-37 (`as u8`)."""
    rows = np.array([[0, 0], [2, 0], [0, 2], [2, 2]], np.uint8)
    init = np.array([[1, 1], [200, 200]], np.uint8)
    cent, iters = oracle.kmeans_lloyd(rows, init, "l2sqr", 5, 1e-6)
    assert cent.tolist() == [[1, 1], [200, 200]] and iters == 1
    rows = np.array([[1, 0], [2, 0]], np.uint8)
    cent, _ = oracle.kmeans_lloyd(rows, np.array([[0, 0]], np.uint8), "l2sqr", 1, 0.0)
    assert cent.tolist() == [[1, 0]]  # mean 1.5 truncates toward zero


def test_result_set_boundary_semantics(oracle):
    """candidate_pair.rs:61-74: k=0 -> empty, k>N -> N, ties keep the lower id in an ascending scan."""
    base = np.zeros((6, 4), np.float32)
    base[3:] = 1.0
    q = np.zeros((1, 4), np.float32)
    ids, dd, cnt = oracle.flat_knn(base, q, 2, "l2sqr")
    assert ids[0].tolist() == [0, 1] and cnt[0] == 2
    ids, dd, cnt = oracle.flat_knn(base, q, 9, "l2sqr")
    assert cnt[0] == 6 and ids[0, :6].tolist() == [0, 1, 2, 3, 4, 5]
    ids, dd, cnt = oracle.flat_knn(base, q, 0, "l2sqr")
    assert cnt[0] == 0


def test_recall(oracle):
    """candidate_pair.rs:127-140."""
    assert oracle.recall([1, 2, 3, 4], [4, 3, 9, 8]) == 0.5


def test_u8_l2_is_an_exact_integer_below_2_pow_24(oracle):
    """The reference casts u8 to f32 and sums (x - q)^2 sequentially in f32 (distance/mod.rs:86-94): every term and,
    below 2^24, every partial sum is an integer, so the reference value IS the exact integer sum. The CUDA path computes
    that integer directly (VABSDIFF4 + IDP.4A, csrc/scanmath.cuh) and converts it once - bit-identical in this range,
    which covers GIST-shaped u8 data (960 dims, values around 18: sums of a few 10^5)."""
    rng = np.random.default_rng(5)
    for dim, hi in ((960, 64), (960, 256), (100, 256), (17, 256)):
        a = rng.integers(0, hi, (50, dim), dtype=np.uint8)
        b = rng.integers(0, hi, (50, dim), dtype=np.uint8)
        exact = ((a.astype(np.int64) - b.astype(np.int64)) ** 2).sum(axis=1)
        for i in range(50):
            d = oracle.distance(a[i], b[i], "l2sqr")
            if exact[i] < (1 << 24):
                assert float(d) == float(exact[i])
            else:   # above 2^24 the sequential f32 sum rounds: still within the parity rule of the exact value
                assert abs(float(d) - float(exact[i])) <= 1e-5 * float(exact[i])


@pytest.mark.parametrize("metric", ["l2sqr", "cosine"])
def test_u8_flat_oracle_equals_numpy_emulation(fixtures, oracle, metric):
    """The reference's other scalar type (Scalar for u8, scalar.rs:39-46; u8 distances cast to f32 first,
    distance/mod.rs:80-94): oracle == independent numpy emulation, bit for bit, on the byte-quantised GIST fixture
    (values x 255, rounded) - 120 queries x 1000 rows x 960 dims, k = 10."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import np_emul as E
    base = np.clip(np.rint(fixtures["base"] * 255.0), 0, 255).astype(np.uint8)
    q = np.clip(np.rint(fixtures["test"][:120] * 255.0), 0, 255).astype(np.uint8)
    ids, dd, cnt = oracle.flat_knn(base, q, 10, metric, os.cpu_count())
    eids, edd = E.flat_knn(base, q, 10, metric)
    assert (cnt == 10).all()
    assert (ids.astype(np.int64) == eids).all()
    assert (bits(dd) == bits(edd)).all()
