"""Tensor-core pruning bounds at their rounding edges.

Every batched search on a shard of >= 65536 rows is exact only because a tensor-core contraction gives each (query, row)
pair a LOWER bound S' of its distance (rows with S' > tau_q are never looked at again) and, for the thresholds, an UPPER
bound U. On smooth random data the margin between the k-th distance and tau_q hides a bound that is wrong by a factor
of two, so these tests put rows exactly where the bounds are tight: BF16 rounding midpoints of PQ lookup tables,
caller-chosen thresholds one ulp above the k-th distance, operands whose rounding or accumulation error is as large as
the bound allows."""
import ctypes as C

import numpy as np
import pytest

from conftest import assert_knn_parity

pytestmark = pytest.mark.gpu

K = 16


@pytest.fixture(scope="module")
def V():
    import lab_1806_vec_db_b200 as V
    return V


def _stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


# ---- PQ: one-hot filter (pq_gemm.cu) and decoded filter (pq_dec.cu) -------------------------------------------------
def _rel_bound(e, m):
    """Relative bound of the one-hot filter with a BF16 unit roundoff of 2^e, in the f32 arithmetic of pq_gemm.cu."""
    return np.float32(np.float32(1.05 * 2.0 ** e) + np.float32(m) * np.float32(2.0 ** -21))


def _bf16(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).to(torch.bfloat16).float().numpy()


def _pack(codes):
    """[n, m] centroid indices -> reference layout (low nibble = even group)."""
    n, m = codes.shape
    c = np.zeros((n, m + (m & 1)), np.uint8)
    c[:, :m] = codes
    return np.ascontiguousarray(c[:, 0::2] | (c[:, 1::2] << 4))


def _table(V, books, codes, dpg, dtype=np.float32):
    """PQ table whose rows ARE the chosen centroids (so the codes are known): books [m, 16, dpg], codes [n, m]."""
    m = books.shape[0]
    base = np.ascontiguousarray(books[np.arange(m)[None, :], codes].reshape(codes.shape[0], m * dpg), dtype)
    vs = V.DeviceVecSet(base, "l2sqr")
    flat = np.ascontiguousarray(books.reshape(-1), dtype)
    pq = V.PQTable(vs, V.PQConfig(4, m, "l2sqr"), flat, codes=_pack(codes))
    return base, vs, flat, pq


# exact ADC: E = 1.004 (one entry just above the BF16 midpoint 1.00390625: rounds up to 1.0078125),
# T = 0.5 + 0.50195 + 0.0025 = 1.00445 (0.50195 just below the midpoint 0.501953125: rounds down to 0.5)
_ET_VALUES = np.r_[0.0, 1.004, 0.5, 0.50195, 0.0025, 4.0 + np.arange(11.0)]


def _et_set(V, m, dpg, n=66_000, seed=0):
    rng = np.random.default_rng(seed + m)
    books = np.zeros((m, 16, dpg), np.float32)
    books[:, :, 0] = np.sqrt(_ET_VALUES).astype(np.float32)      # query 0: the LUT entry is the squared first coordinate
    codes = rng.integers(5, 16, (n, m)).astype(np.uint8)         # background: ADC >= 4 m
    t_rows = np.arange(16, n, 33)                                # ~3 % of every stretch of rows: the sample sees them
    codes[t_rows] = 0
    codes[t_rows, 0], codes[t_rows, 1], codes[t_rows, 2] = 2, 3, 4
    e_rows = np.array([1000, 33_001, 65_990])
    assert not np.isin(e_rows, t_rows).any()
    codes[e_rows] = 0
    codes[e_rows, 0] = 1
    return (*_table(V, books, codes, dpg), codes, t_rows, e_rows)


@pytest.mark.parametrize("m,dpg,no_decode", [(8, 2, None), (7, 2, None), (16, 4, "1"), (16, 4, "0")])
def test_pq_filter_keeps_rows_that_bf16_rounds_up(V, oracle, m, dpg, no_decode, monkeypatch):
    """A row E whose only LUT entry rounds UP in BF16 by almost 2^-8 against ~2000 rows T whose entries round down: with
    a 2^-9 bound, E's S' lands above the threshold the T rows set (the j0-th smallest sampled U), E is dropped and the T
    rows still pass the count check, so the result is silently wrong. The >= 32-query tensor path must return the bits
    of the < 32-query FP32 scan and the oracle's result, E rows first. (m = 16, 4 dims per group: the decoded
    contraction, and the one-hot one under VDB_PQ_NO_DECODE=1.)"""
    from lab_1806_vec_db_b200 import _lib as L
    if no_decode is not None:
        monkeypatch.setenv("VDB_PQ_NO_DECODE", no_decode)
    base, vs, books, pq, codes, t_rows, e_rows = _et_set(V, m, dpg)
    q = np.zeros((40, m * dpg), np.float32)
    # precondition, in the arithmetic of pq_gemm.cu: the data sits between the wrong (2^-9) and the right (2^-8) bound
    lut = pq.create_lookup(q[:1])[0][0]
    adc = pq.adc_distances(q[:1])[0]
    assert adc[e_rows].max() < adc[t_rows].min()
    lb = _bf16(lut)
    s_e = np.float32(sum(np.float64(lb[g * 16 + codes[e_rows[0], g]]) for g in range(m)))
    s_t = np.float32(sum(np.float64(lb[g * 16 + codes[t_rows[0], g]]) for g in range(m)))
    for e, dropped in ((-9, True), (-8, False)):
        lower_e = np.float32(np.float64(s_e) * np.float64(np.float32(1) - _rel_bound(e, m)) - 1e-35)
        upper_t = np.float32(s_t * (np.float32(1) + _rel_bound(e, m)))
        assert (lower_e > upper_t) == dropped, (e, lower_e, upper_t)
    idx = V.FlatIndex(vs)
    lib = L.lib()
    for k, ef in ((10, 40), (5, 100)):
        L.check(lib.vdb_prof_reset())
        L.check(lib.vdb_prof_enable(1))
        try:
            got = idx.knn_pq_batch(q, k, ef, pq)
            ms, launches = C.c_double(0), C.c_uint64(0)
            L.check(lib.vdb_prof_read(b"pq_gemm", C.byref(ms), C.byref(launches)))
        finally:
            L.check(lib.vdb_prof_enable(0))
        assert launches.value >= 2, "the batch did not take the tensor-core filter"
        few = idx.knn_pq_batch(q[:9], k, ef, pq)     # < 32 queries: FP32 global-threshold scan
        assert (few[0] == got[0][:9]).all() and (few[1].view(np.uint32) == got[1][:9].view(np.uint32)).all()
        assert (got[0] == got[0][:1]).all()          # identical queries, identical answers
        assert got[0][0, :3].tolist() == sorted(e_rows.tolist()), got[0][0]
        want = oracle.flat_knn_pq(base, pq.encoded_vec_set, books, m, 4, q[:2], k, ef, "l2sqr", nthreads=8)
        assert_knn_parity(base, q[:2], "l2sqr", tuple(a[:2] for a in got), want, oracle)


def _pq_bounds(pq, q, path):
    import torch
    from lab_1806_vec_db_b200 import _lib as L
    dq = torch.from_numpy(np.ascontiguousarray(q)).cuda()
    n = len(pq.vec_set)
    lower = torch.empty((q.shape[0], n), dtype=torch.float32, device="cuda")
    upper = torch.empty_like(lower)
    L.check(L.lib().vdb_debug_pq_bounds_dev(pq._h, C.c_void_p(dq.data_ptr()), q.shape[0], path, C.c_void_p(lower.data_ptr()),
                                            C.c_void_p(upper.data_ptr()), _stream()))
    return lower.cpu().numpy(), upper.cpu().numpy()


def _assert_bounds(pq, q, path):
    lower, upper = _pq_bounds(pq, q, path)
    adc = pq.adc_distances(q)                        # bit-exact reference ADC
    bad_lo, bad_up = lower > adc, adc > upper
    assert not bad_lo.any(), f"path {path}: S' > adc for {int(bad_lo.sum())} pairs, worst ratio {float((lower / adc)[bad_lo].max())}"
    assert not bad_up.any(), f"path {path}: U < adc for {int(bad_up.sum())} pairs, worst ratio {float((upper / adc)[bad_up].min())}"
    return lower, upper, adc


def _midpoint_books(m, dpg, rng):
    """Centroids whose squared norm (the LUT entry of a zero query) sits 2^-12 above (even index) or below (odd index) a
    BF16 rounding midpoint with a small mantissa, where the relative rounding error is largest; group 0 dominates."""
    j = rng.integers(0, 4, (m, 16))
    e = rng.integers(-2, 3, (m, 16)).astype(np.float64)
    e[0] += 10.0
    mid = 2.0 ** e * (1.0 + (2 * j + 1) * 2.0 ** -8)
    sign = np.where(np.arange(16) % 2 == 0, 1.0, -1.0)[None, :]
    books = np.zeros((m, 16, dpg), np.float32)
    books[:, :, 0] = np.sqrt(mid * (1.0 + sign * 2.0 ** -12)).astype(np.float32)
    return books


@pytest.mark.parametrize("m,dpg", [(8, 2), (16, 4)])
def test_pq_one_hot_bounds_hold_for_every_pair(V, m, dpg):
    """S' <= adc <= U for EVERY (query, row) of the one-hot contraction, with LUT entries just above and just below BF16
    rounding midpoints (a 2^-9 bound fails on both sides), one dominant group and random codes."""
    rng = np.random.default_rng(m)
    n = 66_000
    books = _midpoint_books(m, dpg, rng)
    codes = rng.integers(0, 16, (n, m)).astype(np.uint8)
    _, _, _, pq = _table(V, books, codes, dpg)
    q = np.zeros((64, m * dpg), np.float32)
    q[32:] = rng.standard_normal((32, m * dpg)).astype(np.float32) * np.float32(0.01)   # entries off the midpoints
    lower, upper, adc = _assert_bounds(pq, q, 0)
    # and they are tight: within 2^-6 relative of the exact value (2 x 2^-8: the rounding plus the bound's own margin)
    assert (lower >= adc * (1 - 2.0 ** -6)).all() and (upper <= adc * (1 + 2.0 ** -6)).all()


@pytest.mark.parametrize("qscale", [1.0, 1e3, 1e-3])
def test_pq_decoded_bounds_hold_for_every_pair(V, qscale):
    """The decoded contraction (FP16 centroids and queries, one power-of-two scale each) under codebooks spanning six
    decades and queries scaled by 1e3 / 1e-3: the filter keeps every row at tau = its own adc, and U >= adc."""
    rng = np.random.default_rng(int(qscale * 1000) % 97)
    m, dpg, n = 16, 4, 66_000
    books = (rng.standard_normal((m, 16, dpg)) * 10.0 ** rng.uniform(-3, 3, (m, 16, 1))).astype(np.float32)
    codes = rng.integers(0, 16, (n, m)).astype(np.uint8)
    base, _, _, pq = _table(V, books, codes, dpg)
    q = (rng.standard_normal((64, m * dpg)) * 10.0 ** rng.uniform(-3, 3, (64, 1))).astype(np.float32)
    q[:8] = base[rng.integers(0, n, 8)]              # queries on rows: adc ~ 0 for some pairs
    q = (q * np.float32(qscale)).astype(np.float32)
    _assert_bounds(pq, q, 1)
    _assert_bounds(pq, q, 0)


# ---- Flat: the filter under a tight, caller-chosen threshold (flat_gemm.cu, vdb_tq_* phases) --------------------------
def _shells(rng, n, dim, nq):
    q = (rng.standard_normal((nq, dim)) * 3.0).astype(np.float32)
    per = 64
    u = rng.standard_normal((nq * per, dim))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    r = 1.0 + 1e-5 * rng.uniform(-1, 1, (nq * per, 1))
    base = (rng.standard_normal((n, dim)) * 3.0).astype(np.float32)
    rows = rng.choice(n, nq * per, replace=False)
    base[rows] = (np.repeat(q, per, 0) + r * u).astype(np.float32)
    return base, q


def _offset(rng, n, dim, nq):
    base = (100.0 + 1e-3 * rng.standard_normal((n, dim))).astype(np.float32)
    q = (100.0 + 1e-3 * rng.standard_normal((nq, dim))).astype(np.float32)
    return base, q


def _signs(rng, n, dim, nq):
    """|x_i| = t |q_i| for every row (sum |q_i x_i| = ||q|| ||x||) with random signs (the dot product is a few percent
    of it); operands exact in FP16 and TF32, so the accumulation term is the whole bound."""
    t = (1.0 + rng.integers(0, 8, (n, 1)) * 2.0 ** -10).astype(np.float32)
    base = (rng.choice([-1.0, 1.0], (n, dim)) * t).astype(np.float32)
    q = rng.choice([-1.0, 1.0], (nq, dim)).astype(np.float32) * np.float32(0.75)
    return base, q


def _u8(rng, n, dim, nq):
    return rng.integers(200, 256, (n, 960), dtype=np.uint8), rng.integers(200, 256, (nq, 960), dtype=np.uint8)


def _random(rng, n, dim, nq):
    return rng.random((n, dim), dtype=np.float32), rng.random((nq, dim), dtype=np.float32)


_SETS = {"shells": _shells, "offset": _offset, "signs": _signs, "u8": _u8, "random": _random}
_cache = {}


def _dataset(V, name, metric):
    key = (name, metric)
    if key not in _cache:
        base, q = _SETS[name](np.random.default_rng(len(name)), 66_000, 128, 129)
        _cache.clear()                               # one set on the device at a time
        _cache[key] = (base, q, V.DeviceVecSet(base, metric))
    return _cache[key]


def _scan_keys(vs, dq, k):
    import torch
    from lab_1806_vec_db_b200 import _lib as L
    keys = torch.empty((dq.shape[0], k), dtype=torch.int64, device="cuda")
    L.check(L.lib().vdb_flat_scan_keys_dev(vs._h, C.c_void_p(dq.data_ptr()), dq.shape[0], k, C.c_void_p(keys.data_ptr()),
                                           _stream()))
    torch.cuda.synchronize()
    return keys.cpu().numpy().astype(np.uint64)


def _shifted_tau(q, keys, col, metric):
    """tau_q = nextafter(d - ||q||^2, +inf) (cosine: nextafter(d, +inf)) of the distance in column `col` of the keys."""
    from lab_1806_vec_db_b200.sharded import unpack_keys
    d, _ = unpack_keys(keys[:, col])
    if metric == "cosine":
        return np.nextafter(d.astype(np.float32), np.float32(np.inf))
    q64 = q.astype(np.float64)
    return np.nextafter((d.astype(np.float64) - (q64 * q64).sum(1)).astype(np.float32), np.float32(np.inf))


class _Tq:
    """The tensor-core phases of one batch (vdb_tq_*), as the row-sharded search drives them, without the sample."""

    def __init__(self, vs, dq):
        from lab_1806_vec_db_b200 import _lib as L
        self.L, self.lib, self.nq = L, L.lib(), dq.shape[0]
        self.h = C.c_void_p()
        L.check(self.lib.vdb_tq_begin_dev(vs._h, C.c_void_p(dq.data_ptr()), self.nq, _stream(), C.byref(self.h)))

    def filter(self, k, tau):
        import torch
        dtau = torch.from_numpy(np.ascontiguousarray(tau, np.float32)).cuda()
        keys = torch.empty((self.nq, k), dtype=torch.int64, device="cuda")
        ovf = torch.zeros((self.nq,), dtype=torch.int32, device="cuda")
        self.L.check(self.lib.vdb_tq_filter_dev(self.h, k, C.c_void_p(dtau.data_ptr()), C.c_void_p(keys.data_ptr()),
                                                C.c_void_p(ovf.data_ptr())))
        torch.cuda.synchronize()
        return keys.cpu().numpy().astype(np.uint64), ovf.cpu().numpy()

    def check(self, keys, k, n, tau):
        import torch
        dk = torch.from_numpy(np.ascontiguousarray(keys).view(np.int64)).cuda()
        dtau = torch.from_numpy(np.ascontiguousarray(tau, np.float32)).cuda()
        ovf = torch.zeros((self.nq,), dtype=torch.int32, device="cuda")
        redo = torch.empty((self.nq,), dtype=torch.int32, device="cuda")
        nredo = torch.zeros((1,), dtype=torch.int32, device="cuda")
        self.L.check(self.lib.vdb_tq_check_dev(self.h, C.c_void_p(dk.data_ptr()), k, n, C.c_void_p(dtau.data_ptr()),
                                               C.c_void_p(ovf.data_ptr()), C.c_void_p(redo.data_ptr()),
                                               C.c_void_p(nredo.data_ptr())))
        torch.cuda.synchronize()
        return np.sort(redo.cpu().numpy()[:int(nredo.item())])

    def close(self):
        self.lib.vdb_tq_end(self.h)


@pytest.mark.parametrize("nq", [128, 129])
@pytest.mark.parametrize("kind", ["tf32", "f16"])
@pytest.mark.parametrize("metric", ["l2sqr", "cosine"])
@pytest.mark.parametrize("name", ["shells", "offset", "signs", "u8"])
def test_flat_filter_under_tight_threshold_equals_scan(V, name, metric, kind, nq, monkeypatch):
    """With tau_q one ulp above the k-th exact distance (shifted by ||q||^2 for L2Sqr), every row of the true top-k sits
    right at the threshold: a lower bound that is wrong anywhere drops one of them. The filter (contraction, upper-bound
    pruning, exact rerank) must return the exact scan's keys bit for bit for every query whose list did not overflow;
    single CTAs (128 queries) and CTA pairs (129)."""
    import torch
    if name == "u8" and kind == "tf32":
        pytest.skip("u8 rows always feed the contraction as FP16 (exact for bytes)")
    monkeypatch.setenv("VDB_GEMM_KIND", kind)
    base, q, vs = _dataset(V, name, metric)
    q = q[:nq]
    dq = torch.from_numpy(np.ascontiguousarray(q)).cuda()
    scan = _scan_keys(vs, dq, K)
    tau = _shifted_tau(q, scan, K - 1, metric)
    tq = _Tq(vs, dq)
    try:
        keys, ovf = tq.filter(K, tau)
    finally:
        tq.close()
    ok = ovf == 0
    if name != "offset":                             # the offset set is below the operands' resolution: lists overflow
        assert ok.mean() > 0.9, f"{int((~ok).sum())} of {nq} lists overflowed"
    bad = np.nonzero(ok & (keys != scan).any(1))[0]
    assert bad.size == 0, f"queries {bad[:10].tolist()} differ from the scan ({bad.size} of {int(ok.sum())})"


@pytest.mark.parametrize("kind", ["tf32", "f16"])
@pytest.mark.parametrize("metric", ["l2sqr", "cosine"])
def test_flat_check_flags_exactly_the_unproven_queries(V, metric, kind, monkeypatch):
    """The completeness check of the exact top-k keys: with tau_q at the (k/2)-th true distance no query is provably
    complete, on near-equidistant shells too (its slack must not let d_k through); with tau_q at the 4k-th on random data
    every query is."""
    import torch
    monkeypatch.setenv("VDB_GEMM_KIND", kind)
    for name in ("shells", "random"):
        base, q, vs = _dataset(V, name, metric)
        dq = torch.from_numpy(np.ascontiguousarray(q)).cuda()
        scan = _scan_keys(vs, dq, 4 * K)
        tq = _Tq(vs, dq)
        try:
            half = tq.check(scan[:, :K].copy(), K, len(base), _shifted_tau(q, scan, K // 2 - 1, metric))
            far = tq.check(scan[:, :K].copy(), K, len(base), _shifted_tau(q, scan, 4 * K - 1, metric))
        finally:
            tq.close()
        assert half.tolist() == list(range(q.shape[0])), (name, half.size)
        if name == "random":
            assert far.size == 0, (name, far[:10].tolist())


# ---- IVF: the probe scan in table mode ------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["shells", "offset"])
def test_ivf_probe_scan_at_rounding_edges_equals_fp32_scan(V, name):
    """Near-equidistant shells and a large common offset through the tensor probe scan (>= 16 queries): ids and distance
    bits equal the FP32 list scan (< 16 queries)."""
    base, q, vs = _dataset(V, name, "l2sqr")
    rng = np.random.default_rng(3)
    cent = np.concatenate([q[:24], base[rng.choice(len(base), 8, replace=False)]])
    ivf = V.IVFIndex(vs, cent)
    for k, nprobe in ((K, 2), (100, 6)):
        got = ivf.knn_with_ef_batch(q[:40], k, nprobe)
        for lo in (0, 9, 18):
            fp32 = ivf.knn_with_ef_batch(q[lo:lo + 9], k, nprobe)
            assert (fp32[0] == got[0][lo:lo + 9]).all(), (k, nprobe, lo)
            assert (fp32[1].view(np.uint32) == got[1][lo:lo + 9].view(np.uint32)).all()
            assert (fp32[2] == got[2][lo:lo + 9]).all()
