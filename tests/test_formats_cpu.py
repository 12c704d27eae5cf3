"""`not gpu`: on-disk formats either side of the path (bincode 1.3.3 layouts, raw vectors, fvecs, bench TOML)."""
import struct

import numpy as np
import pytest

from lab_1806_vec_db_b200 import formats as F


def test_ground_truth_known_bytes():
    """Vec<GroundTruthRow{Vec<usize>}>: u64 count, then per row u64 len + u64 ids (candidate_pair.rs:111-191)."""
    data = F.dump_ground_truth([[3, 1], [7]])
    assert data == struct.pack("<QQQQQQ", 2, 2, 3, 1, 1, 7)
    rows = F.load_ground_truth(data)
    assert [r.tolist() for r in rows] == [[3, 1], [7]]
    assert F.recall(rows[0], [1, 9, 3]) == 1.0 and F.recall([1, 2, 3, 4], [4, 3, 9, 8]) == 0.5
    with pytest.raises(ValueError):
        F.load_ground_truth(data + b"\0")


def test_flat_index_file_is_the_distance_tag():
    assert F.dump_flat_index("l2sqr") == b"\x00\x00\x00\x00" and F.dump_flat_index("cosine") == b"\x01\x00\x00\x00"
    assert F.load_flat_index(b"\x01\x00\x00\x00") == "cosine"


def test_kmeans_record_known_bytes():
    """KMeans{config{k,max_iter,tol,dist,selected: Option<Range>}, centroids: VecSet{dim,data}}."""
    km = F.KMeansRecord(2, 20, 1e-6, "cosine", (4, 6), np.array([[1, 2], [3, 4]], np.float32))
    w = F._W()
    F._w_kmeans(w, km, np.float32)
    want = (struct.pack("<QQfI", 2, 20, 1e-6, 1) + b"\x01" + struct.pack("<QQ", 4, 6) +
            struct.pack("<QQ", 2, 4) + struct.pack("<4f", 1, 2, 3, 4))
    assert bytes(w.b) == want
    back = F._r_kmeans(F._R(want), np.float32)
    assert back.selected == (4, 6) and back.dist == "cosine" and back.centroids.tolist() == [[1, 2], [3, 4]]
    w = F._W()
    F._w_kmeans(w, km._replace(selected=None), np.float32)
    assert bytes(w.b)[24:25] == b"\x00"  # Option::None tag right after k, max_iter, tol, dist


def test_pq_table_round_trip_and_header_layout():
    rng = np.random.default_rng(0)
    groups = [F.KMeansRecord(16, 20, 1e-6, "l2sqr", (3 * g, 3 * g + 3), rng.random((16, 3), dtype=np.float32))
              for g in range(5)]
    rec = F.PQTableRecord(4, 5, "l2sqr", 100, 20, 1e-6, 15, rng.integers(0, 256, (7, 3), dtype=np.uint8), groups,
                          np.zeros(80, np.float32))
    data = F.dump_pq_table(rec)
    # PQConfig{n_bits, m, dist, k_means_size: Some(100), max_iter, tol}, dim, k, encoded_dim
    head = struct.pack("<QQI", 4, 5, 0) + b"\x01" + struct.pack("<Q", 100) + struct.pack("<Qf", 20, 1e-6)
    head += struct.pack("<QQQ", 15, 16, 3)
    assert data.startswith(head)
    back = F.load_pq_table(data)
    assert (back.encoded_vec_set == rec.encoded_vec_set).all() and back.k_means_size == 100
    assert all((a.centroids == b.centroids).all() and a.selected == b.selected for a, b in zip(back.group_k_means, groups))
    assert F.dump_pq_table(back) == data


def test_ivf_index_round_trip_without_vec_set():
    rng = np.random.default_rng(1)
    km = F.KMeansRecord(3, 20, 1e-6, "l2sqr", None, rng.random((3, 8), dtype=np.float32))
    rec = F.IVFIndexRecord("l2sqr", 4, np.zeros((0, 8), np.float32), 3, 100, 20, 1e-6,
                           [np.array([0, 4]), np.array([], np.uint64), np.array([1, 2, 3])], km)
    data = F.dump_ivf_index(rec, dim=8)
    assert data.startswith(struct.pack("<IQQQ", 0, 4, 8, 0))  # dist, default_n_probes, VecSet{dim=8, data=[]}
    back = F.load_ivf_index(data)
    assert back.vec_set.shape == (0, 8) and [c.tolist() for c in back.clusters] == [[0, 4], [], [1, 2, 3]]
    assert F.dump_ivf_index(back, dim=8) == data


def test_raw_and_fvecs(tmp_path, fixtures):
    p = tmp_path / "v.bin"
    F.save_raw(p, fixtures["base"][:5])
    assert (F.load_raw(p, 960) == fixtures["base"][:5]).all()
    assert F.load_raw(p, 960, limit=2).shape == (2, 960)
    with pytest.raises(ValueError):
        F.load_raw(p, 7)
    rows = np.arange(12, dtype=np.float32).reshape(3, 4)
    with open(tmp_path / "v.fvecs", "wb") as f:
        for r in rows:
            f.write(struct.pack("<i", 4) + r.tobytes())
    assert (F.read_fvecs(tmp_path / "v.fvecs") == rows).all()


# BenchConfig / ResultList files in the reference's layout (examples/bench.rs:70-92, 312-368), carrying the settings and
# published numbers of config/bench_10000_ivf.toml, config/bench_pq_240_hnsw.toml and data/t_bench_1e4.toml that
# BASELINE.md and bench_configs.py quote
BENCH_CONFIG = """label = "{label}"
dist = "L2Sqr"
gnd_path = "data/gnd_{label}.bin"
index_cache = "data/index_{label}.bin"
bench_output = "data/t_bench.toml"

[ef.range]
start = {ef0}
end = {ef1}
step = {step}

[algorithm.{algo}]
{body}
{pq}
[base]
dim = 960
data_type = "float32"
data_path = "data/base.bin"

[test]
dim = 960
data_type = "float32"
data_path = "data/test.bin"
"""
RESULT_LIST = """title = "Bench (N=10000)"

[[results]]
label = "HNSW"
ef = [120, 360]
search_time = [0.0382, 0.0816]
recall = [0.9927, 0.9990]

[[results]]
label = "HNSW+PQ"
ef = [160, 360]
search_time = [0.0369, 0.0632]
recall = [0.9930, 0.9989]

[[results]]
label = "Flat+PQ"
ef = [100, 200]
search_time = [0.1271, 0.1360]
recall = [0.9915, 0.9997]
"""


def test_reference_files_parse(tmp_path, fixtures):
    """The reference's data file (rebuilt bit for bit from the fixture) and config / result files in its layout load
    through these readers."""
    import hashlib
    F.save_raw(tmp_path / "gist_1000.bin", fixtures["base"])
    assert hashlib.sha256((tmp_path / "gist_1000.bin").read_bytes()).hexdigest() == fixtures["base_sha256"]
    base = F.load_raw(tmp_path / "gist_1000.bin", 960)
    assert base.shape == (1000, 960) and (base[50] == base[444]).all()
    (tmp_path / "ivf.toml").write_text(BENCH_CONFIG.format(
        label="IVF", ef0=8, ef1=24, step=4, algo="IVF", pq="",
        body="k = 128\nk_means_size = 1000\nk_means_max_iter = 20\nk_means_tol = 1e-6"))
    cfg = F.load_bench_config(tmp_path / "ivf.toml")
    assert cfg["ef_values"] == [8, 12, 16, 20, 24] and cfg["algorithm"]["IVF"]["k"] == 128 and cfg["dist"] == "l2sqr"
    (tmp_path / "pq.toml").write_text(BENCH_CONFIG.format(
        label="HNSW+PQ", ef0=240, ef1=600, step=60, algo="HNSW", body="ef_construction = 200\nM = 16",
        pq='[PQ]\ndist = "L2Sqr"\nn_bits = 4\nm = 240\nk_means_size = 10000\nk_means_max_iter = 20\nk_means_tol = 1e-6\n'))
    cfg = F.load_bench_config(tmp_path / "pq.toml")
    assert cfg["PQ"]["m"] == 240 and cfg["ef_values"] == list(range(240, 601, 60))
    res = F.load_result_list(RESULT_LIST)
    assert [r["label"] for r in res["results"]][:2] == ["HNSW", "HNSW+PQ"]
    text = F.dump_result_list(res["title"], res["results"])
    again = F.load_result_list(text)
    assert again["title"] == res["title"] and again["results"][0]["ef"] == res["results"][0]["ef"]
    assert np.allclose(again["results"][2]["search_time"], res["results"][2]["search_time"])


def test_hnsw_index_bincode_layout_known_answer():
    """HNSWIndex serde (hnsw_index.rs:99-141): field order of the struct, usize -> u64, Option tag u8, Vec = u64 len +
    items, dist_cache skipped; byte-level check of a 2-node graph and a round trip."""
    import struct
    from lab_1806_vec_db_b200 import formats as F
    rec = F.HNSWIndexRecord(dim=3, dist="cosine", max_elements=2, m=2, max_m0=4, ef_construction=4, default_ef=2,
                            inv_log_m=1.4426950216293335, start_batch_since=1000,
                            vec_set=np.zeros((0, 3), np.float32),
                            level0_links=np.array([1, 0, 0, 0, 0, 0, 0, 0], np.uint32),
                            other_links=[np.array([1, 0], np.uint32), np.zeros(0, np.uint32)],
                            links_len=[np.array([1, 0], np.uint64), np.array([1], np.uint64)],
                            vec_level=np.array([1, 0], np.uint64), num_deleted=0, enter_level=1, enter_point=0)
    data = F.dump_hnsw_index(rec)
    head = struct.pack("<QIQQQQQfQ", 3, 1, 2, 2, 4, 4, 2, 1.4426950216293335, 1000)   # HNSWInnerConfig, Cosine = tag 1
    assert data[:len(head)] == head
    o = len(head)
    assert data[o:o + 16] == struct.pack("<QQ", 3, 0)                                   # VecSet {dim, data: []}
    o += 16
    assert data[o:o + 8] == struct.pack("<Q", 8) and data[o + 8:o + 12] == struct.pack("<I", 1)
    tail = struct.pack("<Q", 0) + b"\x01" + struct.pack("<Q", 1) + b"\x01" + struct.pack("<Q", 0)
    assert data.endswith(tail)                                                          # num_deleted, Some(1), Some(0)
    back = F.load_hnsw_index(data)
    assert back.dist == "cosine" and back.m == 2 and back.enter_level == 1 and back.enter_point == 0
    assert (back.level0_links == rec.level0_links).all() and (back.vec_level == rec.vec_level).all()
    assert [a.tolist() for a in back.other_links] == [[1, 0], []]
    assert [a.tolist() for a in back.links_len] == [[1, 0], [1]]
    empty = F.load_hnsw_index(F.dump_hnsw_index(rec._replace(enter_level=None, enter_point=None)))
    assert empty.enter_level is None and empty.enter_point is None


def test_load_raw_limit_ignores_a_trailing_partial_row(tmp_path):
    """BinaryScalar::from_binary_file reads at most limit * dim scalars (scalar.rs:78-98): bytes beyond them - even a
    partial row - are never examined; without a limit the same file is rejected (vec_set.rs:35-38)."""
    from lab_1806_vec_db_b200 import formats as F
    rows = np.arange(5 * 8, dtype=np.float32).reshape(5, 8)
    p = tmp_path / "x.bin"
    with open(p, "wb") as f:
        f.write(rows.tobytes())
        f.write(np.zeros(3, np.float32).tobytes())        # a trailing partial row
    got = F.load_raw(p, 8, np.float32, limit=4)
    assert got.shape == (4, 8) and (got == rows[:4]).all()
    with pytest.raises(ValueError):
        F.load_raw(p, 8, np.float32)
