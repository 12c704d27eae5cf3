"""8-bit and long-sub-vector PQ through every encode and ADC scan path.

The golden PQ tests cover 4-bit codes on sub-vectors of at most 8 dimensions. Here every other branch of pq.cu runs at
least once and is checked stage by stage against the reference arithmetic, bit for bit: the generic encoder
(pq_encode_kernel: 8-bit codes, 4-bit sub-vectors longer than 8, tables too large for the staged encoder), the per-CTA
ADC scan with 1, 2 or 4 queries per pass and the lookup tables in shared memory or read through L1, the 8-bit word loop
with a partial last word, the top-k under the highest candidate pressure the scan allows, the batched 8-bit training
and its per-group fallback, row-sharded 8-bit tables and the 8-bit file round trip.

Every case names the branch it is meant to take and asserts it as a precondition (`_plan` mirrors `adc_scan`), so a
change of the kernel's constants fails loudly instead of moving a case off its branch."""
import ctypes as C
import sys

import numpy as np
import pytest

from conftest import GOLDEN, assert_knn_parity

pytestmark = pytest.mark.gpu

if GOLDEN not in sys.path:
    sys.path.insert(0, GOLDEN)
import np_emul as E  # noqa: E402

KEY_NONE = np.uint64(0xFFFFFFFFFFFFFFFF)
NQS = (1, 2, 3, 5, 9)                     # ragged last query group of a pass for every NQ


@pytest.fixture(scope="module")
def V():
    import lab_1806_vec_db_b200 as V
    return V


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


# ---- mirrors of the kernels' launch decisions (pq.cu, kmeans.cu) ---------------------------------------------------
ADC_THREADS = 512                         # pq.cu: ADC_THREADS
ADC_SMEM_MAX = 200 * 1024                 # pq.cu: ADC_SMEM_MAX
ENC_MAXL, ENC_ROWS = 8, 8                 # pq.cu: ENC_MAXL, ENC_ROWS


def _next_pow2(x):
    return 1 << (int(x) - 1).bit_length()


def _plan(m, n_bits, metric, K, nq):
    """(NQ, lut_smem, smem bytes, P) that adc_scan picks for nq queries; K = 0 is the all-distances mode of
    adc_distances (no top-k segments). Raises ValueError where adc_scan rejects the shape."""
    tab = m << n_bits
    cosine = metric == "cosine"
    P = _next_pow2(K + 2 * ADC_THREADS) if K else 0      # topk_segment_size(K, ADC_THREADS)

    def smem(t, ls):
        s = (t * tab + (tab if cosine else 0)) * 4 if ls else 0
        return s + (t * P * 8 + t * 4 if K else 0)         # TopkSmem::bytes(t, P)

    nqt = 4
    while nqt > 1 and nqt >> 1 >= nq:
        nqt >>= 1
    while nqt > 1 and smem(nqt, True) > ADC_SMEM_MAX:
        nqt >>= 1
    ls = smem(nqt, True) <= ADC_SMEM_MAX
    if smem(nqt, ls) > ADC_SMEM_MAX:
        raise ValueError(f"ef={K} too large for the fused top-k")
    return nqt, ls, smem(nqt, ls), P


def _iters(n, smem, sms):
    """Row tiles each CTA of the per-CTA scan visits (grid = one wave at the occupancy shared memory allows)."""
    tiles = -(-n // ADC_THREADS)
    occ = max(1, min(8, (220 * 1024) // max(smem, 1)))
    grid = max(1, min(tiles, sms * occ))
    return -(-tiles // grid), grid


def _encoder(n_bits, m, max_len, dim):
    """pq_create's choice: the staged 4-bit encoder or the generic pq_encode_kernel."""
    mp = m + (m & 1)
    smem4 = (max_len * 16 * mp + 16 * mp + ENC_ROWS * ((dim + 3) & ~3)) * 4 + mp * 4
    fast = n_bits == 4 and max_len <= ENC_MAXL and smem4 <= 200 * 1024 and dim < 65536
    return "encode4" if fast else "generic"


def _train_batched(kc, max_len):
    """kmeans.cu: pq_train_supported."""
    return kc <= 256 and kc * max_len * 8 + kc * 8 <= 160 * 1024


def test_plan_mirror_thresholds():
    """The 8-bit thresholds of adc_scan at ef <= 1024: L2Sqr 4 / 2 / 1 queries per pass up to m = 33 / 83 / 183, cosine
    (which also stages dist_cache) up to 27 / 55 / 91, then the L1 path; 4-bit reaches L1 at m = 2944."""
    def last(metric, n_bits, want):
        return max(m for m in range(1, 4000) if _plan(m, n_bits, metric, 64, 9)[:2] == want)
    assert [last("l2sqr", 8, (t, True)) for t in (4, 2, 1)] == [33, 83, 183]
    assert [last("cosine", 8, (t, True)) for t in (4, 2, 1)] == [27, 55, 91]
    assert last("l2sqr", 4, (1, True)) == 2943 and _plan(2944, 4, "l2sqr", 64, 9)[:2] == (1, False)
    with pytest.raises(ValueError):
        _plan(16, 8, "l2sqr", 15361, 1)


# ---- reference computations ----------------------------------------------------------------------------------------
def _order_keys(adc, kk):
    """Top-kk keys by (order bits of the f32 ADC value, id), KEY_NONE padded: what the scan must select."""
    d = np.asarray(adc, np.float32) + np.float32(0.0)
    b = d.view(np.uint32)
    o = np.where(b & 0x80000000, ~b, b | np.uint32(0x80000000)).astype(np.uint64)
    keys = np.sort((o << np.uint64(32)) | np.arange(len(d), dtype=np.uint64))
    out = np.full(kk, KEY_NONE, np.uint64)
    out[:min(kk, len(keys))] = keys[:kk]
    return out


class _Ref:
    """The oracle's lookup tables and the sequential-f32 emulation of the ADC sums (tests/golden/np_emul.py)."""

    def __init__(self, oracle, codes, books, dim, m, n_bits, metric):
        self.o, self.codes, self.books = oracle, codes, books
        self.m, self.n_bits, self.metric = m, n_bits, metric
        self.dc = oracle.pq_dist_cache(dim, books, m, n_bits, metric)
        self._adc = {}

    def lookup(self, q):
        return self.o.pq_lookup(q, self.books, self.m, self.n_bits, self.metric)

    def adc(self, q):
        key = q.tobytes()
        if key not in self._adc:
            lut, qc = self.lookup(q)
            self._adc[key] = E.pq_adc(self.codes, self.m, self.n_bits, lut, self.dc, qc, self.metric)
        return self._adc[key]


def _adc_keys(vs, pq, q, kk):
    """vdb_pq_adc_keys_dev: the shard's top-kk (ADC, id) keys, before the rerank."""
    import torch
    from lab_1806_vec_db_b200 import _lib as L
    dq = torch.from_numpy(np.ascontiguousarray(q)).cuda()
    keys = torch.empty((q.shape[0], kk), dtype=torch.int64, device="cuda")
    L.check(L.lib().vdb_pq_adc_keys_dev(vs._h, pq._h, C.c_void_p(dq.data_ptr()), q.shape[0], kk,
                                        C.c_void_p(keys.data_ptr()), _stream()))
    torch.cuda.synchronize()
    return keys.cpu().numpy().view(np.uint64)


def _launches(fn, *names):
    """(result of fn(), {kernel name: launches}) from the library's profiling counters."""
    from lab_1806_vec_db_b200 import _lib as L
    lib = L.lib()
    L.check(lib.vdb_prof_reset())
    L.check(lib.vdb_prof_enable(1))
    try:
        out = fn()
        counts = {}
        for name in names:
            ms, n = C.c_double(0), C.c_uint64(0)
            L.check(lib.vdb_prof_read(name.encode(), C.byref(ms), C.byref(n)))
            counts[name] = n.value
    finally:
        L.check(lib.vdb_prof_enable(0))
    return out, counts


def _same(a, b):
    assert (a[0] == b[0]).all() and (bits(a[1]) == bits(b[1])).all() and (a[2] == b[2]).all()


def _books(rows, m, kc, dup_every=3):
    """Codebooks taken from kc data rows (rows 100..100+kc). In every `dup_every`-th group centroid kc-2 repeats
    centroid 1, and row 101 sits on both: its encode ties and must go to the lower id."""
    parts = []
    for g, (lo, hi) in enumerate(E.pq_groups(rows.shape[1], m)):
        c = np.array(rows[100:100 + kc, lo:hi])
        if g % dup_every == 0:
            c[kc - 2] = c[1]
        parts.append(c.reshape(-1))
    return np.ascontiguousarray(np.concatenate(parts))


def _check_stages(V, oracle, base, q, books, m, n_bits, metric, vs, pq, kks=(40, 2000), nq_e2e=3,
                  sweep=((10, 4), (10, 64), (5, None), (10, 2000)), code_rows=20_000):
    """Codes, LUT + qcache, every ADC value, the selected candidate keys and the reranked result, against the
    oracle and the sequential-f32 emulation. Returns the (NQ, lut_smem) branches the scans took."""
    n, dim = base.shape
    codes = pq.encoded_vec_set
    ref = _Ref(oracle, codes, books, dim, m, n_bits, metric)
    # codes
    assert (codes[:code_rows] == oracle.pq_encode(base[:code_rows], books, m, n_bits, metric, nthreads=8)).all()
    # lookup tables and query norms
    lut, qc = pq.create_lookup(q)
    for i in range(len(q)):
        wl, wq = ref.lookup(q[i])
        assert (bits(lut[i]) == bits(wl)).all(), f"query {i}: LUT"
        assert bits(qc[i]) == bits(np.float32(wq)), f"query {i}: qcache"
    # every ADC value, nq in NQS: ragged query groups for every NQ
    taken = set()
    for nq in NQS:
        taken.add(_plan(m, n_bits, metric, 0, nq)[:2])
        adc = pq.adc_distances(q[:nq])
        for i in range(nq):
            want = ref.adc(q[i])
            bad = np.nonzero(bits(adc[i]) != bits(want))[0]
            assert bad.size == 0, f"nq={nq} query {i}: {bad.size} ADC values differ, first row {bad[0]}"
    rows = np.random.default_rng(0).choice(n, 24, replace=False)
    for i in range(2):                                        # the oracle's own ADC on a few rows
        lut_i, qc_i = ref.lookup(q[i])
        want = oracle.pq_adc(codes[rows], m, n_bits, metric, lut_i, ref.dc, qc_i)
        assert (bits(ref.adc(q[i])[rows]) == bits(want)).all()
    # the candidate set: exactly the top-max(ef, k) keys by (ADC, id)
    for kk in kks:
        want = np.stack([_order_keys(ref.adc(q[i]), kk) for i in range(len(q))])
        for nq in NQS:
            taken.add(_plan(m, n_bits, metric, kk, nq)[:2])
            got = _adc_keys(vs, pq, q[:nq], kk)
            bad = np.nonzero((got != want[:nq]).any(1))[0]
            assert bad.size == 0, f"kk={kk} nq={nq}: queries {bad.tolist()} select other candidates"
    # end to end: ef < k, ef > n, a large ef with a larger top-k segment
    idx = V.FlatIndex(vs)
    for k, ef in sweep:
        ef = n + 50 if ef is None else ef
        got = idx.knn_pq_batch(q, k, ef, pq)
        want = oracle.flat_knn_pq(base, codes, books, m, n_bits, q[:nq_e2e], k, ef, metric, nthreads=8)
        assert_knn_parity(base, q[:nq_e2e], metric, tuple(a[:nq_e2e] for a in got), want, oracle)
        one = idx.knn_pq_batch(q[-1:], k, ef, pq)             # NQ = 1 for the same query
        _same(one, tuple(a[-1:] for a in got))
    return taken


# ---- 8-bit codes and long 4-bit sub-vectors, small shards ----------------------------------------------------------
# (name, n_bits, metric, dtype, n, dim, m, encoder, per-CTA branch at ef <= 1024 and 9 queries)
CASES = [
    ("b8-l2-m18-nq4", 8, "l2sqr", np.float32, 14_000, 90, 18, "generic", (4, True)),
    ("b8-l2-m47-nq2", 8, "l2sqr", np.float32, 12_000, 160, 47, "generic", (2, True)),
    ("b8-l2-m121-nq1", 8, "l2sqr", np.float32, 8_000, 420, 121, "generic", (1, True)),
    ("b8-l2-m241-l1", 8, "l2sqr", np.float32, 6_000, 600, 241, "generic", (1, False)),
    ("b8-cos-m18-nq4", 8, "cosine", np.float32, 14_000, 60, 18, "generic", (4, True)),
    ("b8-cos-m47-nq2", 8, "cosine", np.float32, 12_000, 120, 47, "generic", (2, True)),
    ("b8-cos-m90-nq1", 8, "cosine", np.float32, 8_000, 300, 90, "generic", (1, True)),
    ("b8-cos-m121-l1", 8, "cosine", np.float32, 6_000, 500, 121, "generic", (1, False)),
    ("b8-u8-l2-m30-nq4", 8, "l2sqr", np.uint8, 10_000, 100, 30, "generic", (4, True)),
    ("b8-u8-cos-m61-nq1", 8, "cosine", np.uint8, 10_000, 190, 61, "generic", (1, True)),
    ("b4-l2-len16", 4, "l2sqr", np.float32, 8_000, 128, 8, "generic", (4, True)),
    ("b4-cos-len16", 4, "cosine", np.float32, 8_000, 128, 8, "generic", (4, True)),
    ("b4-l2-len14-15", 4, "l2sqr", np.float32, 8_000, 100, 7, "generic", (4, True)),
    ("b4-cos-len14-15", 4, "cosine", np.float32, 8_000, 100, 7, "generic", (4, True)),
    ("b4-l2-len8", 4, "l2sqr", np.float32, 8_000, 64, 8, "encode4", (4, True)),
    ("b4-l2-len9", 4, "l2sqr", np.float32, 8_000, 72, 8, "generic", (4, True)),
    ("b4-l2-len1-dim3000-l1", 4, "l2sqr", np.float32, 3_000, 3000, 3000, "generic", (1, False)),
]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_pq_stages_bit_exact(V, oracle, case):
    """Every stage against the reference arithmetic on the branch the case is named for; m % 4 != 0 for every 8-bit
    case (a partial last code word), uneven groups, duplicated centroids (encode ties to the lowest id)."""
    name, n_bits, metric, dtype, n, dim, m, encoder, branch = case
    groups = E.pq_groups(dim, m)
    max_len = max(hi - lo for lo, hi in groups)
    assert _encoder(n_bits, m, max_len, dim) == encoder
    assert _plan(m, n_bits, metric, 40, 9)[:2] == branch, _plan(m, n_bits, metric, 40, 9)
    rng = np.random.default_rng(len(name) * 1000 + m)
    if dtype == np.uint8:
        base = rng.integers(0, 256, (n, dim), dtype=np.uint8)
        q = rng.integers(0, 256, (9, dim), dtype=np.uint8)
    else:
        base = rng.random((n, dim), dtype=np.float32)
        q = rng.random((9, dim), dtype=np.float32)
    base[3000:3040] = base[101]                      # rows on the duplicated centroids: encode ties, ADC ties by id
    q[0] = base[101]
    kc = 1 << n_bits
    books = _books(base, m, kc)
    vs = V.DeviceVecSet(base, metric)
    pq = V.PQTable(vs, V.PQConfig(n_bits, m, metric), books)
    assert pq.encoded_vec_set.shape == (n, m if n_bits == 8 else (m + 1) // 2)
    taken = _check_stages(V, oracle, base, q, books, m, n_bits, metric, vs, pq)
    assert branch in taken


def test_pq_ef_beyond_the_fused_top_k_is_an_error(V):
    """Known gap: the per-CTA scan holds max(ef, k) + 1024 candidates per query in shared memory, so ef > 15 360 is
    refused with a VdbError (the reference accepts any ef). Pinned so that the limit stays an error, not a wrong
    answer."""
    rng = np.random.default_rng(3)
    base = rng.random((20_000, 32), dtype=np.float32)
    vs = V.DeviceVecSet(base, "l2sqr")
    pq = V.PQTable(vs, V.PQConfig(8, 16, "l2sqr"), _books(base, 16, 256))
    idx = V.FlatIndex(vs)
    with pytest.raises(ValueError):
        _plan(16, 8, "l2sqr", 15_361, 1)
    with pytest.raises(V.VdbError, match="too large for the fused top-k"):
        idx.knn_pq_batch(base[:1], 10, 15_361, pq)
    got = idx.knn_pq_batch(base[:1], 10, 15_360, pq)      # the largest ef the scan takes
    assert got[2][0] == 10 and got[0][0, 0] == 0


# ---- large shards --------------------------------------------------------------------------------------------------
def test_pq_8bit_batch_on_a_large_shard_stays_on_the_per_cta_scan(V, oracle):
    """8-bit codes on a shard >= 65 536 rows: the global-threshold scan and the tensor-core filter take 4-bit codes
    only, so a batch of 40 queries runs the per-CTA scan (one launch) and equals the queries sent one at a time."""
    rng = np.random.default_rng(8)
    n, dim, m = 66_000, 48, 16
    base = rng.random((n, dim), dtype=np.float32)
    base[5000:5200] = base[101]
    q = rng.random((40, dim), dtype=np.float32)
    q[0] = base[101]
    books = _books(base, m, 256)
    vs = V.DeviceVecSet(base, "l2sqr")
    pq = V.PQTable(vs, V.PQConfig(8, m, "l2sqr"), books)
    assert (pq.encoded_vec_set[:20_000] == oracle.pq_encode(base[:20_000], books, m, 8, "l2sqr", nthreads=8)).all()
    idx = V.FlatIndex(vs)
    for k, ef in ((10, 100), (5, 1500)):
        got, c = _launches(lambda: idx.knn_pq_batch(q, k, ef, pq), "pq_adc", "pq_gemm")
        assert c == {"pq_adc": 1, "pq_gemm": 0}, c
        for i in range(len(q)):
            _same(idx.knn_pq_batch(q[i:i + 1], k, ef, pq), tuple(a[i:i + 1] for a in got))
        want = oracle.flat_knn_pq(base, pq.encoded_vec_set, books, m, 8, q[:4], k, ef, "l2sqr", nthreads=8)
        assert_knn_parity(base, q[:4], "l2sqr", tuple(a[:4] for a in got), want, oracle)


def test_pq_long_groups_large_shard_three_paths(V, oracle):
    """4-bit codes on 16-dimension sub-vectors (pq_groups(128, 8)) on a shard >= 65 536 rows: the per-CTA scan
    (< 4 queries), the global-threshold FP32 scan (4-31) and the one-hot BF16 filter (>= 32) return the same ids and
    distance bits, and the oracle's result."""
    rng = np.random.default_rng(16)
    n, dim, m = 66_000, 128, 8
    base = rng.random((n, dim), dtype=np.float32)
    base[5000:5300] = base[101]
    q = rng.random((40, dim), dtype=np.float32)
    q[0] = base[101]
    books = _books(base, m, 16)
    vs = V.DeviceVecSet(base, "l2sqr")
    pq = V.PQTable(vs, V.PQConfig(4, m, "l2sqr"), books)
    assert (pq.encoded_vec_set[:20_000] == oracle.pq_encode(base[:20_000], books, m, 4, "l2sqr", nthreads=8)).all()
    idx = V.FlatIndex(vs)
    for k, ef in ((10, 50), (10, 300), (5, 1200)):
        tensor, c = _launches(lambda: idx.knn_pq_batch(q, k, ef, pq), "pq_gemm")
        assert c["pq_gemm"] >= 2, "the batch did not take the tensor-core filter"
        fp32, c = _launches(lambda: idx.knn_pq_batch(q[:9], k, ef, pq), "pq_adc", "pq_gemm")
        assert c["pq_gemm"] == 0 and c["pq_adc"] >= 2, c
        cta, c = _launches(lambda: idx.knn_pq_batch(q[:3], k, ef, pq), "pq_adc", "pq_gemm")
        assert c == {"pq_adc": 1, "pq_gemm": 0}, c
        _same(fp32, tuple(a[:9] for a in tensor))
        _same(cta, tuple(a[:3] for a in tensor))
        want = oracle.flat_knn_pq(base, pq.encoded_vec_set, books, m, 4, q[:3], k, ef, "l2sqr", nthreads=8)
        assert_knn_parity(base, q[:3], "l2sqr", cta, want, oracle)


# ---- adversarial code orders ---------------------------------------------------------------------------------------
def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _adversarial(V, oracle, n_bits, m, n, order, seed):
    """Rows that ARE their centroids (1-2 dimensions per group, distinct centroids), codes chosen so that the ADC of
    query 0 DESCENDS with the row id (every row beats every row before it) or all codes are identical (every ADC
    ties). The table is built from the codes; a fresh encode of the rows must give them back."""
    rng = np.random.default_rng(seed)
    kc = 1 << n_bits
    dim = m if n_bits == 8 else 2 * m
    perm = np.argsort(rng.random((m, kc)), axis=1)   # distinct first coordinates: a row's own centroid is unique
    books = (rng.random((m, kc, dim // m)) * 0.5 + perm[:, :, None]).astype(np.float32)
    codes_idx = rng.integers(0, kc, (n, m))
    if order == "same":
        codes_idx[:] = codes_idx[0]
    q = (rng.random((9, dim)) * kc).astype(np.float32)
    flat = np.ascontiguousarray(books.reshape(-1))
    if order == "desc":
        lut = oracle.pq_lookup(q[0], flat, m, n_bits, "l2sqr")[0].reshape(m, kc)
        adc = E.seq_sum(lut[np.arange(m)[None, :], codes_idx])
        codes_idx = codes_idx[np.lexsort((np.arange(n), -adc.astype(np.float64)))]
    base = np.ascontiguousarray(books[np.arange(m)[None, :], codes_idx].reshape(n, dim))
    codes = codes_idx.astype(np.uint8) if n_bits == 8 else np.ascontiguousarray(
        (codes_idx[:, 0::2] | (codes_idx[:, 1::2] << 4)).astype(np.uint8))
    vs = V.DeviceVecSet(base, "l2sqr")
    pq = V.PQTable(vs, V.PQConfig(n_bits, m, "l2sqr"), flat, codes=codes)
    fresh = V.PQTable(vs, V.PQConfig(n_bits, m, "l2sqr"), flat)
    assert (fresh.encoded_vec_set == codes).all()
    fresh.close()
    if order == "desc":
        a = pq.adc_distances(q[:1])[0]
        assert (np.diff(a.astype(np.float64)) <= 0).all()
    return base, q, flat, codes, vs, pq


def _pressure(m, n_bits, K, n):
    """The per-CTA scan must reach its flush limit more than once: every CTA visits >= 3 row tiles and, with every
    row of a tile pushed, a segment flushed only at P - K (no room for one more tile) would overflow."""
    nqt, ls, smem, P = _plan(m, n_bits, "l2sqr", K, 1)
    it, _ = _iters(n, smem, _sms())
    assert it >= 3 and (P - K) < it * ADC_THREADS and (P - K) // ADC_THREADS + 1 <= it, (it, P, K)
    return ls


@pytest.mark.parametrize("order", ["desc", "same"])
@pytest.mark.parametrize("n_bits", [8, 4])
def test_pq_adversarial_code_orders(V, oracle, n_bits, order):
    """Rows in descending ADC order push every row into the per-CTA top-k, which flushes at the highest rate the
    kernel allows; all-identical codes tie every ADC, so the order is by id alone. The shard holds 3 row tiles per
    CTA of the widest grid (>= 65 536 rows), so 4-bit batches also run the global-threshold scan (9 queries) and
    the tensor-core filter (40), whose candidate lists overflow on the tied codes and are redone per CTA."""
    sms = _sms()
    m = 100 if n_bits == 8 else 16                    # 8-bit: a 100 KB LUT keeps one CTA per SM, at K = 1000 too
    n = 3 * sms * ADC_THREADS
    base, q, books, codes, vs, pq = _adversarial(V, oracle, n_bits, m, n, order, 40 + n_bits)
    ref = _Ref(oracle, codes, books, base.shape[1], m, n_bits, "l2sqr")
    pressure = [15_000] + ([1000] if n_bits == 8 else [])
    branches = {_pressure(m, n_bits, K, n) for K in pressure}
    if n_bits == 8:
        assert branches == {True, False}             # the LUT in shared memory (K = 1000) and through L1 (15 000)
    qb = np.ascontiguousarray(np.concatenate([np.repeat(q[:1], 20, 0), q[1:], np.repeat(q[:1], 12, 0)]))   # 40
    adc = pq.adc_distances(q)
    for i in range(len(q)):
        assert (bits(adc[i]) == bits(ref.adc(q[i]))).all(), f"query {i}: ADC"
    want = {}
    for kk in (10, 1000, 15_000):
        for i in range(len(q)):
            want[(kk, i)] = _order_keys(ref.adc(q[i]), kk)
        if order == "same":
            assert (want[(kk, 0)] >> np.uint64(32) == want[(kk, 0)][0] >> np.uint64(32)).all()
        for nq in (1, 3, 9, 40):
            qs = q[:nq] if nq <= 9 else qb
            got = _adc_keys(vs, pq, qs, kk)
            for j in range(nq):
                i = j if nq <= 9 else (0 if j < 20 or j >= 28 else j - 19)
                assert (got[j] == want[(kk, i)]).all(), f"kk={kk} nq={nq} query {j}: other candidates"
    idx = V.FlatIndex(vs)
    for k, ef in ((10, 1), (10, 1000), (10, 15_000)):
        ref_one = idx.knn_pq_batch(q[:1], k, ef, pq)
        for qs in (q[:3], q, qb):                   # every copy of query 0 in a batch gets the single query's bits
            got = idx.knn_pq_batch(qs, k, ef, pq)
            for j in np.nonzero((qs == q[0]).all(1))[0]:
                _same(tuple(a[j:j + 1] for a in got), ref_one)
        want_knn = oracle.flat_knn_pq(base, codes, books, m, n_bits, q[:2], k, ef, "l2sqr", nthreads=8)
        assert_knn_parity(base, q[:2], "l2sqr", tuple(a[:2] for a in idx.knn_pq_batch(q, k, ef, pq)), want_knn, oracle)
        if order == "same":
            assert ref_one[0][0].tolist() == list(range(k))


# ---- batched training, 8-bit ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("metric", ["l2sqr", "cosine"])
@pytest.mark.parametrize("dtype", [np.float32, np.uint8])
def test_batched_pq_training_8bit_bit_exact_vs_per_group(V, oracle, metric, dtype):
    """kc = 256 in one launch: given the same initial codebooks the result equals the per-group Lloyd and the oracle
    bit for bit, with duplicated initial centroids (the higher id stays empty and keeps its centroid)."""
    from lab_1806_vec_db_b200.index import train_codebooks
    rng = np.random.default_rng(256)
    n, dim, m = 1500, 21, 8
    rows = (rng.random((n, dim)) * (255 if dtype == np.uint8 else 1)).astype(dtype)
    rows[100:400] = rows[7]
    assert _train_batched(256, max(hi - lo for lo, hi in E.pq_groups(dim, m)))
    cfg = V.PQConfig(8, m, metric, None, 8, 1e-6)
    vs = V.DeviceVecSet(rows, metric)
    init, parts = [], []
    for lo, hi in V.pq_groups(dim, m):
        ini = np.ascontiguousarray(rows[rng.permutation(n)[:256], lo:hi])
        ini[200:210] = ini[3]                            # duplicated centroids: empty clusters from the first pass
        init.append(ini.reshape(-1))
        km = V.KMeans.from_vec_set(vs, V.KMeansConfig(256, 8, 1e-6, metric, (lo, hi)), rng, ini)
        want, _ = oracle.kmeans_lloyd(rows, ini, metric, 8, 1e-6, sel=(lo, hi))
        assert (np.asarray(want).reshape(-1).view(np.uint8) == km.centroids.reshape(-1).view(np.uint8)).all()
        parts.append(km.centroids.reshape(-1))
    got = train_codebooks(vs, cfg, rng, np.concatenate(init))
    assert (got.view(np.uint8) == np.concatenate(parts).view(np.uint8)).all()


def test_pq_training_8bit_long_groups_take_the_per_group_path(V, oracle):
    """kc = 256 on sub-vectors of 80 dimensions does not fit one CTA: vdb_pq_train_ds refuses it with
    VDB_EUNSUPPORTED and train_codebooks trains group by group, with the same bits as the oracle."""
    from lab_1806_vec_db_b200 import _lib as L
    from lab_1806_vec_db_b200.index import train_codebooks
    rng = np.random.default_rng(80)
    n, dim, m = 700, 160, 2
    rows = rng.random((n, dim), dtype=np.float32)
    assert not _train_batched(256, 80)
    vs = V.DeviceVecSet(rows, "l2sqr")
    init = [np.ascontiguousarray(rows[rng.permutation(n)[:256], lo:hi]) for lo, hi in V.pq_groups(dim, m)]
    for ini in init:
        ini[100] = ini[5]
    flat = np.ascontiguousarray(np.concatenate([i.reshape(-1) for i in init]))
    out = np.zeros_like(flat)
    it = np.zeros(m, np.uint32)
    rc = L.lib().vdb_pq_train_ds(vs._h, m, 8, 5, 1e-6, None, L.ptr(flat), L.ptr(out), L.ptr(it))
    assert rc == L.EUNSUPPORTED
    got = train_codebooks(vs, V.PQConfig(8, m, "l2sqr", None, 5, 1e-6), rng, flat)
    want = np.concatenate([oracle.kmeans_lloyd(rows, ini, "l2sqr", 5, 1e-6, sel=(lo, hi))[0].reshape(-1)
                           for ini, (lo, hi) in zip(init, V.pq_groups(dim, m))])
    assert (got.view(np.uint32) == want.view(np.uint32)).all()


# ---- row-sharded 8-bit tables and the file round trip --------------------------------------------------------------
def _device_sets():
    import torch
    sets = [[0, 0, 0]]
    if torch.cuda.device_count() >= 2:
        sets.append(list(range(min(torch.cuda.device_count(), 4))))
    return sets


@pytest.mark.parametrize("metric", ["l2sqr", "cosine"])
def test_sharded_8bit_pq_equals_the_unsharded_table(V, oracle, metric):
    """vdb_pq_create / vdb_pq_knn with 8-bit codes on a row-sharded set: codes and results bit-identical to the
    unsharded table; adc_distances has no sharded implementation and says so."""
    rng = np.random.default_rng(3 if metric == "l2sqr" else 4)
    n, dim, m = 30_000, 60, 23
    base = rng.random((n, dim), dtype=np.float32)
    base[20_001] = base[101]                         # a duplicate in another shard: the lower id first
    q = rng.random((12, dim), dtype=np.float32)
    q[0] = base[101]
    books = _books(base, m, 256)
    cfg = V.PQConfig(8, m, metric)
    try:
        V.init_devices([])
        full_vs = V.DeviceVecSet(base, metric)
        full = V.PQTable(full_vs, cfg, books)
        idx = V.FlatIndex(full_vs)
        sweep = ((10, 100), (10, 4), (3, 2000))
        want = {s: idx.knn_pq_batch(q, s[0], s[1], full) for s in sweep}
        codes = full.encoded_vec_set
        for devs in _device_sets():
            V.init_devices(devs)
            vs = V.DeviceVecSet(base, metric)
            assert [d for d, _, _ in vs.shards()] == devs
            pq = V.PQTable(vs, cfg, books)
            assert (pq.encoded_vec_set == codes).all()
            flat = V.FlatIndex(vs)
            for (k, ef), w in want.items():
                _same(flat.knn_pq_batch(q, k, ef, pq), w)
                _same(flat.knn_pq_batch(q[:1], k, ef, pq), tuple(a[:1] for a in w))
            with pytest.raises(V.VdbError):
                pq.adc_distances(q[:1])
            del pq, flat, vs
    finally:
        V.init_devices([])
    o = oracle.flat_knn_pq(base, codes, books, m, 8, q[:3], 10, 100, metric, nthreads=8)
    assert_knn_parity(base, q[:3], metric, tuple(a[:3] for a in want[(10, 100)]), o, oracle)


@pytest.mark.parametrize("metric", ["l2sqr", "cosine"])
def test_8bit_table_file_round_trip(V, oracle, metric):
    """An 8-bit table written in the reference's PQTable layout, read back and loaded from its codes searches
    bit-identically to the freshly encoded table."""
    from lab_1806_vec_db_b200 import formats as F
    rng = np.random.default_rng(9)
    n, dim, m = 8_000, 100, 47
    base = rng.random((n, dim), dtype=np.float32)
    q = rng.random((5, dim), dtype=np.float32)
    books = _books(base, m, 256)
    vs = V.DeviceVecSet(base, metric)
    pq = V.PQTable(vs, V.PQConfig(8, m, metric), books)
    rec = F.load_pq_table(F.dump_pq_table(F.pq_table_record(pq)))
    assert rec.n_bits == 8 and rec.m == m and rec.encoded_vec_set.shape == (n, m)
    assert (bits(rec.dist_cache) == bits(oracle.pq_dist_cache(dim, books, m, 8, metric))).all()
    loaded_books = np.concatenate([km.centroids.reshape(-1) for km in rec.group_k_means])
    assert (bits(loaded_books) == bits(books)).all()
    loaded = V.PQTable(vs, V.PQConfig(rec.n_bits, rec.m, rec.dist), loaded_books, codes=rec.encoded_vec_set)
    assert (bits(loaded.adc_distances(q)) == bits(pq.adc_distances(q))).all()
    idx = V.FlatIndex(vs)
    for k, ef in ((10, 60), (5, 600)):
        _same(idx.knn_pq_batch(q, k, ef, loaded), idx.knn_pq_batch(q, k, ef, pq))
