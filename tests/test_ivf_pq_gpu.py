"""IVF + PQ search (IVFIndex.knn_pq / vdb_ivf_knn_pq, csrc/ivf_pq.cu) against the IVF knn_pq reference (ivf_pq_reference.py).

Definition (INTEGRATION.md): FlatIndex::knn_pq restricted to the rows of the n_probes nearest lists. The candidate keys
(ADC, id) are BIT-EXACT against the oracle; the reranked results follow the parity rule; with every list probed the result
is bit-identical to FlatIndex.knn_pq_batch on the same table."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import assert_knn_parity
from ivf_pq_reference import ivf_knn_pq

pytestmark = pytest.mark.gpu

NT = os.cpu_count() or 1
SHAPES = [("pq240", 240, 4, 960), ("pq7", 7, 4, 13), ("pq5b8", 5, 8, 13)]
SWEEP = ((10, 240), (10, 4), (3, 2000))


@pytest.fixture(scope="module")
def V():
    import lab_1806_vec_db_b200 as V
    yield V
    V.init_devices([])


def _same(got, want):
    assert (np.asarray(got[0]).astype(np.int64) == np.asarray(want[0]).astype(np.int64)).all()
    assert (np.asarray(got[1]).view(np.uint32) == np.asarray(want[1]).view(np.uint32)).all()
    assert (np.asarray(got[2]) == np.asarray(want[2])).all()


def _keys_of(ids, adc, counts):
    """The library's packed (distance, id) keys of the oracle's candidate lists, UINT64_MAX padded."""
    b = (np.asarray(adc, np.float32) + np.float32(0)).view(np.uint32).astype(np.uint64)   # -0 -> +0
    o = np.where(b & 0x80000000, ~b & 0xFFFFFFFF, b | 0x80000000)
    keys = (o << np.uint64(32)) | np.asarray(ids, np.uint64)
    keys[np.arange(keys.shape[1])[None, :] >= np.asarray(counts)[:, None]] = np.iinfo(np.uint64).max
    return keys


def _adc_keys(V, vs, ivf, pq, queries, kk, n_probes):
    import torch
    q = torch.from_numpy(np.ascontiguousarray(queries)).cuda()
    out = torch.empty((queries.shape[0], kk), dtype=torch.int64, device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    V._lib.check(V.lib().vdb_ivf_pq_adc_keys_dev(vs._h, ivf._h, pq._h, C.c_void_p(q.data_ptr()), queries.shape[0], kk,
                                                 n_probes, C.c_void_p(out.data_ptr()), st))
    torch.cuda.synchronize()
    return out.cpu().numpy().view(np.uint64)


def _books(V, rows, m, n_bits, first=0):
    """Codebooks from data rows: group g = rows[first : first + 2^n_bits, lo:hi]."""
    kc = 1 << n_bits
    return np.concatenate([np.ascontiguousarray(rows[first:first + kc, lo:hi]).reshape(-1)
                           for lo, hi in V.pq_groups(rows.shape[1], m)])


class Case:
    """A set, its IVF index and PQ table on the GPU, and the same lists / codes for the oracle."""

    def __init__(self, V, oracle, base, cent, books, m, n_bits, metric):
        self.base, self.cent, self.books, self.m, self.n_bits, self.metric = base, cent, books, m, n_bits, metric
        self.vs = V.DeviceVecSet(base, metric)
        self.ivf = V.IVFIndex(self.vs, cent)
        self.pq = V.PQTable(self.vs, V.PQConfig(n_bits, m, metric), books)
        self.codes = oracle.pq_encode(base, books, m, n_bits, metric, nthreads=NT)
        assert (self.pq.encoded_vec_set == self.codes).all()
        assign = oracle.kmeans_assign(base, cent, metric, nthreads=NT)
        assert (self.ivf.assignment == assign).all()
        self.off, self.mem = oracle.ivf_lists(assign, cent.shape[0])

    def oracle(self, oracle, queries, k, ef, n_probes, candidates=False):
        want, cand = ivf_knn_pq(oracle, self.base, self.codes, self.books, self.m, self.n_bits, self.cent, self.off,
                                self.mem, queries, k, ef, n_probes, self.metric)
        return (want, cand) if candidates else want

    def check(self, V, oracle, queries, k, ef, n_probes):
        """Candidate keys bit-exact, final result by the parity rule; returns the final result."""
        want, (ci, cd, cc) = self.oracle(oracle, queries, k, ef, n_probes, candidates=True)
        kk = max(k, ef)
        got_keys = _adc_keys(V, self.vs, self.ivf, self.pq, queries, kk, n_probes)
        assert (got_keys == _keys_of(ci, cd, cc)).all(), f"candidate keys differ (k={k}, ef={ef}, n_probes={n_probes})"
        got = self.ivf.knn_pq_batch(queries, k, ef, self.pq, n_probes)
        assert_knn_parity(self.base, queries, self.metric, got, want, oracle)
        return got


def _golden_case(V, oracle, fixtures, golden, tag, m, n_bits, dimclip, metric):
    base = np.ascontiguousarray(fixtures["base"][:, :dimclip])
    return Case(V, oracle, base, np.ascontiguousarray(base[7:23]), golden[f"{tag}_codebooks"], m, n_bits, metric)


@pytest.mark.parametrize("tag,m,n_bits,dimclip", SHAPES)
@pytest.mark.parametrize("metric", ["l2sqr", "cosine"])
def test_golden_shapes_vs_oracle(V, fixtures, golden, oracle, tag, m, n_bits, dimclip, metric):
    """gist_1000, nlist 16: keys bit-exact, results by the parity rule, over n_probes and (k, ef) incl. ef < k and
    fewer probed rows than k / than max(ef, k)."""
    case = _golden_case(V, oracle, fixtures, golden, tag, m, n_bits, dimclip, metric)
    queries = np.ascontiguousarray(fixtures["test"][:8, :dimclip])
    for n_probes in (1, 4, 16, 50):
        for k, ef in SWEEP:
            case.check(V, oracle, queries, k, ef, n_probes)
    # the trait call: default_n_probes (4)
    pairs = case.ivf.knn_pq(queries[0], 10, 40, case.pq)
    ids, dist, cnt = case.ivf.knn_pq_batch(queries[:1], 10, 40, case.pq, 4)
    assert [p.index for p in pairs] == ids[0, :cnt[0]].tolist()


@pytest.mark.parametrize("metric", ["l2sqr", "cosine"])
def test_all_lists_probed_equals_flat_knn_pq(V, fixtures, golden, oracle, metric):
    case = _golden_case(V, oracle, fixtures, golden, "pq240", 240, 4, 960, metric)
    queries = np.ascontiguousarray(fixtures["test"][:32])
    flat = V.FlatIndex(case.vs)
    for k, ef in SWEEP:
        want = flat.knn_pq_batch(queries, k, ef, case.pq)
        for n_probes in (16, 1000):
            _same(case.ivf.knn_pq_batch(queries, k, ef, case.pq, n_probes), want)


@pytest.mark.parametrize("tag,m,n_bits,dimclip,metric", [("pq240", 240, 4, 960, "l2sqr"), ("pq5b8", 5, 8, 13, "cosine")])
def test_batch_invariance(V, fixtures, golden, oracle, tag, m, n_bits, dimclip, metric):
    """Full and partial query groups per item: every batch gives per query the bits of the nq = 1 call."""
    case = _golden_case(V, oracle, fixtures, golden, tag, m, n_bits, dimclip, metric)
    queries = np.ascontiguousarray(fixtures["test"][:300, :dimclip])
    single = [case.ivf.knn_pq_batch(queries[i:i + 1], 10, 60, case.pq, 4) for i in range(300)]
    for nq in (1, 2, 3, 4, 5, 9, 300):
        got = case.ivf.knn_pq_batch(queries[:nq], 10, 60, case.pq, 4)
        for i in range(nq):
            _same(tuple(a[i:i + 1] for a in got), single[i])


@pytest.mark.parametrize("n_bits", [8, 4])
@pytest.mark.parametrize("metric", ["l2sqr", "cosine"])
def test_u8_rows(V, fixtures, oracle, n_bits, metric):
    base = np.ascontiguousarray(np.clip(fixtures["base"][:, :60] * 255, 0, 255).astype(np.uint8))
    queries = np.ascontiguousarray(np.clip(fixtures["test"][:8, :60] * 255, 0, 255).astype(np.uint8))
    case = Case(V, oracle, base, np.ascontiguousarray(base[7:23]), _books(V, base, 30, n_bits, 300), 30, n_bits, metric)
    for n_probes in (1, 4, 16):
        for k, ef in SWEEP:
            case.check(V, oracle, queries, k, ef, n_probes)


def test_large_set_lists_split_into_ranges(V, oracle):
    """100 000 x 64, nlist 128, m = 16 4-bit, 200 queries at nprobe 8: lists split into several position ranges and
    items start inside a 32-position block. Keys bit-exact against the oracle on a 16-query sample."""
    rng = np.random.default_rng(3)
    n, dim = 100_000, 64
    proto = rng.random((256, dim), dtype=np.float32)
    base = (proto[rng.integers(0, 256, n)] + 0.05 * rng.standard_normal((n, dim), dtype=np.float32)).astype(np.float32)
    queries = (proto[rng.integers(0, 256, 200)] + 0.05 * rng.standard_normal((200, dim), dtype=np.float32)).astype(np.float32)
    cent = np.ascontiguousarray(base[rng.permutation(n)[:128]])
    case = Case(V, oracle, base, cent, _books(V, base, 16, 4, 1000), 16, 4, "l2sqr")
    want, (ci, cd, cc) = case.oracle(oracle, queries[:16], 10, 240, 8, candidates=True)
    keys = _adc_keys(V, case.vs, case.ivf, case.pq, queries, 240, 8)
    assert (keys[:16] == _keys_of(ci, cd, cc)).all()
    got = case.ivf.knn_pq_batch(queries, 10, 240, case.pq, 8)
    assert_knn_parity(base, queries[:16], "l2sqr", tuple(a[:16] for a in got), want, oracle)
    _same(tuple(a[:1] for a in got), case.ivf.knn_pq_batch(queries[:1], 10, 240, case.pq, 8))


def test_edges_empty_list_k0_nq0_and_dev_entry(V, fixtures, golden, oracle):
    import torch
    base = np.ascontiguousarray(fixtures["base"][:, :13])
    cent = np.ascontiguousarray(np.concatenate([base[7:22], np.full((1, 13), 1e6, np.float32)]))   # list 15 stays empty
    case = Case(V, oracle, base, cent, golden["pq7_codebooks"], 7, 4, "l2sqr")
    assert case.off[15] == case.off[16]
    queries = np.ascontiguousarray(np.concatenate([fixtures["test"][:6, :13], np.full((1, 13), 1e6, np.float32)]))
    for n_probes in (1, 2, 16):
        got = case.check(V, oracle, queries, 10, 40, n_probes)
    assert got[2][6] == 10
    got = case.ivf.knn_pq_batch(queries, 10, 40, case.pq, 1)
    assert got[2][6] == 0 and (got[0][6] == np.iinfo(np.uint64).max).all() and np.isnan(got[1][6]).all()
    ids, dist, cnt = case.ivf.knn_pq_batch(queries, 0, 40, case.pq, 4)
    assert ids.shape == (7, 0) and (cnt == 0).all()
    ids, dist, cnt = case.ivf.knn_pq_batch(queries[:0], 10, 40, case.pq, 4)
    assert ids.shape == (0, 10) and cnt.shape == (0,)
    # the device entry point equals the host one
    want = case.ivf.knn_pq_batch(queries, 10, 40, case.pq, 2)
    q = torch.from_numpy(queries).cuda()
    d_ids = torch.empty((7, 10), dtype=torch.int64, device="cuda")
    d_dist = torch.empty((7, 10), dtype=torch.float32, device="cuda")
    d_cnt = torch.empty((7,), dtype=torch.int32, device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    V._lib.check(V.lib().vdb_ivf_knn_pq_dev(case.vs._h, case.ivf._h, case.pq._h, C.c_void_p(q.data_ptr()), 7, 10, 40, 2,
                                            C.c_void_p(d_ids.data_ptr()), C.c_void_p(d_dist.data_ptr()),
                                            C.c_void_p(d_cnt.data_ptr()), st))
    torch.cuda.synchronize()
    _same((d_ids.cpu().numpy(), d_dist.cpu().numpy(), d_cnt.cpu().numpy().astype(np.uint32)), want)


def test_two_tables_on_one_index_and_errors(V, fixtures, golden, oracle):
    """The list-ordered codes are rebuilt when a call brings another table; stale tables / indexes, a metric mismatch
    and n_probes = 0 are errors."""
    base = np.ascontiguousarray(fixtures["base"][:, :13])
    queries = np.ascontiguousarray(fixtures["test"][:8, :13])
    cent = np.ascontiguousarray(base[7:23])
    vs = V.DeviceVecSet(base, "l2sqr")
    ivf = V.IVFIndex(vs, cent)
    off, mem = oracle.ivf_lists(oracle.kmeans_assign(base, cent, "l2sqr", nthreads=NT), 16)
    tables = []
    for tag, m, n_bits in (("pq7", 7, 4), ("pq5b8", 5, 8)):
        books = golden[f"{tag}_codebooks"]
        codes = oracle.pq_encode(base, books, m, n_bits, "l2sqr", nthreads=NT)
        want, _ = ivf_knn_pq(oracle, base, codes, books, m, n_bits, cent, off, mem, queries, 10, 40, 4, "l2sqr")
        tables.append((V.PQTable(vs, V.PQConfig(n_bits, m, "l2sqr"), books), want))
    first = [ivf.knn_pq_batch(queries, 10, 40, pq, 4) for pq, _ in tables]
    for _ in range(2):
        for (pq, want), f in zip(tables, first):
            got = ivf.knn_pq_batch(queries, 10, 40, pq, 4)
            assert_knn_parity(base, queries, "l2sqr", got, want, oracle)
            _same(got, f)
    pq = tables[0][0]
    with pytest.raises(ValueError, match="Distance algorithm mismatch"):
        ivf.knn_pq_batch(queries, 10, 40, V.PQTable(vs, V.PQConfig(4, 7, "cosine"), golden["pq7_codebooks"]), 4)
    with pytest.raises(ValueError, match="greater than 0"):
        ivf.knn_pq_batch(queries, 10, 40, pq, 0)
    vs.push(base[:3])   # the reference drops the PQ table on every write (metadata_vec_table.rs:65)
    with pytest.raises(V.VdbError, match="IVF index was built for a different vector set"):
        ivf.knn_pq(queries[0], 10, 40, pq)
    ivf2 = V.IVFIndex(vs, cent)
    with pytest.raises(V.VdbError, match="PQ table was built for a different vector set"):
        ivf2.knn_pq(queries[0], 10, 40, pq)


def _device_sets():
    import torch
    sets = [[0, 0, 0]]
    if torch.cuda.device_count() >= 2:
        sets.append(list(range(min(torch.cuda.device_count(), 4))))
    return sets


@pytest.mark.parametrize("metric", ["l2sqr", "cosine"])
def test_sharded_set_equals_the_unsharded_call(V, oracle, metric):
    rng = np.random.default_rng(5)
    n, dim, nq = 30_001, 32, 64
    proto = rng.random((64, dim), dtype=np.float32)
    base = (proto[rng.integers(0, 64, n)] + 0.05 * rng.standard_normal((n, dim), dtype=np.float32)).astype(np.float32)
    queries = (proto[rng.integers(0, 64, nq)] + 0.05 * rng.standard_normal((nq, dim), dtype=np.float32)).astype(np.float32)
    cent = np.ascontiguousarray(base[rng.permutation(n)[:32]])
    books = _books(V, base, 8, 4, 500)
    cfg = V.PQConfig(4, 8, metric)
    V.init_devices([])
    vs = V.DeviceVecSet(base, metric)
    ivf, pq = V.IVFIndex(vs, cent), V.PQTable(vs, cfg, books)
    settings = [(10, 240, 1), (10, 240, 4), (3, 600, 8), (10, 5, 32)]
    want = {s: ivf.knn_pq_batch(queries, s[0], s[1], pq, s[2]) for s in settings}
    try:
        for devs in _device_sets():
            V.init_devices(devs)
            vs_s = V.DeviceVecSet(base, metric)
            ivf_s, pq_s = V.IVFIndex(vs_s, cent), V.PQTable(vs_s, cfg, books)
            for s, w in want.items():
                _same(ivf_s.knn_pq_batch(queries, s[0], s[1], pq_s, s[2]), w)
            del ivf_s, pq_s, vs_s
    finally:
        V.init_devices([])
    codes = oracle.pq_encode(base, books, 8, 4, metric, nthreads=NT)
    off, mem = oracle.ivf_lists(oracle.kmeans_assign(base, cent, metric, nthreads=NT), 32)
    o, _ = ivf_knn_pq(oracle, base, codes, books, 8, 4, cent, off, mem, queries[:16], 10, 240, 4, metric)
    assert_knn_parity(base, queries[:16], metric, tuple(a[:16] for a in want[(10, 240, 4)]), o, oracle)
