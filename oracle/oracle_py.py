"""ctypes binding of oracle/liboracle.so (see oracle.h for the reference citations).

TEST INFRASTRUCTURE: the checker, never the thing measured or shipped.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

L2SQR, COSINE = 0, 1
F32, U8 = 0, 1
_METRIC = {"l2sqr": L2SQR, "cosine": COSINE, L2SQR: L2SQR, COSINE: COSINE}


def build():
    subprocess.run(["make", "-s", "-C", _HERE], check=True)


def lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(_HERE, "liboracle.so")
        if not os.path.exists(path):
            build()
        L = C.CDLL(path)
        f, vp, sz, i32 = C.c_float, C.c_void_p, C.c_size_t, C.c_int
        L.orc_dot.restype = f
        L.orc_dot.argtypes = [vp, vp, sz, i32]
        L.orc_l2_sqr.restype = f
        L.orc_l2_sqr.argtypes = [vp, vp, sz, i32]
        L.orc_vec_norm.restype = f
        L.orc_vec_norm.argtypes = [vp, sz, i32]
        L.orc_distance.restype = f
        L.orc_distance.argtypes = [vp, vp, sz, i32, i32]
        L.orc_distance_cached.restype = f
        L.orc_distance_cached.argtypes = [vp, vp, sz, i32, i32, f, f]
        L.orc_dist_cache.restype = f
        L.orc_dist_cache.argtypes = [vp, sz, i32, i32]
        L.orc_flat_knn.argtypes = [vp, sz, sz, i32, i32, vp, sz, sz, vp, vp, vp, i32]
        L.orc_pq_groups.argtypes = [sz, sz, vp]
        L.orc_find_nearest.restype = C.c_uint64
        L.orc_find_nearest.argtypes = [vp, vp, sz, sz, sz, i32, i32]
        L.orc_find_n_nearest.restype = sz
        L.orc_find_n_nearest.argtypes = [vp, vp, sz, sz, i32, i32, sz, vp]
        L.orc_kmeans_assign.argtypes = [vp, sz, sz, i32, i32, vp, sz, sz, sz, vp, i32]
        L.orc_kmeans_lloyd.argtypes = [vp, sz, sz, i32, i32, vp, sz, sz, sz, sz, f]
        L.orc_kmeans_pp_init.argtypes = [vp, sz, sz, i32, i32, sz, sz, sz, C.c_uint64, vp]
        L.orc_kmeans_pp_weights.argtypes = [vp, sz, sz, i32, i32, vp, sz, sz, vp, i32]
        L.orc_pq_encode.argtypes = [vp, sz, sz, i32, i32, vp, sz, sz, vp, i32]
        L.orc_pq_lookup.argtypes = [vp, sz, i32, i32, vp, sz, sz, vp, vp]
        L.orc_pq_dist_cache.argtypes = [sz, i32, i32, vp, sz, sz, vp]
        L.orc_pq_adc.restype = f
        L.orc_pq_adc.argtypes = [vp, sz, sz, i32, vp, vp, f]
        L.orc_flat_knn_pq.argtypes = [vp, sz, sz, i32, i32, vp, vp, sz, sz, vp, sz, sz, sz, vp, vp, vp, i32]
        L.orc_flat_adc_topk.argtypes = [sz, i32, vp, sz, sz, vp, vp, f, sz, vp, vp, vp]
        L.orc_ivf_lists.argtypes = [vp, sz, sz, vp, vp]
        L.orc_ivf_knn.argtypes = [vp, sz, sz, i32, i32, vp, sz, vp, vp, vp, sz, sz, sz, vp, vp, vp, i32]
        L.orc_gather_dist.argtypes = [vp, sz, i32, i32, vp, vp, f, vp, sz, vp]
        L.orc_recall.restype = f
        L.orc_recall.argtypes = [vp, sz, vp, sz]
        _LIB = L
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _dt(a):
    if a.dtype == np.float32:
        return F32
    if a.dtype == np.uint8:
        return U8
    raise TypeError(f"unsupported dtype {a.dtype}")


def _c(a, dtype=None):
    return np.ascontiguousarray(a, dtype=dtype)


def ncores():
    return os.cpu_count() or 1


def distance(a, b, metric):
    a, b = _c(a), _c(b)
    return lib().orc_distance(_p(a), _p(b), a.size, _dt(a), _METRIC[metric])


def dot(a, b):
    a, b = _c(a), _c(b)
    return lib().orc_dot(_p(a), _p(b), a.size, _dt(a))


def dist_cache(a, metric):
    a = _c(a)
    return lib().orc_dist_cache(_p(a), a.size, _dt(a), _METRIC[metric])


def distance_cached(a, b, metric, ca, cb):
    a, b = _c(a), _c(b)
    return lib().orc_distance_cached(_p(a), _p(b), a.size, _dt(a), _METRIC[metric], ca, cb)


def flat_knn(base, queries, k, metric, nthreads=1):
    base, queries = _c(base), _c(queries)
    n, dim = base.shape
    nq = queries.shape[0]
    ids = np.zeros((nq, k), np.uint64)
    dd = np.zeros((nq, k), np.float32)
    cnt = np.zeros(nq, np.uint32)
    rc = lib().orc_flat_knn(_p(base), n, dim, _dt(base), _METRIC[metric], _p(queries), nq, k,
                            _p(ids), _p(dd), _p(cnt), nthreads)
    assert rc == 0
    return ids, dd, cnt


def pq_groups(dim, m):
    out = np.zeros((m, 2), np.uint64)
    rc = lib().orc_pq_groups(dim, m, _p(out))
    assert rc == 0, "pq_groups: invalid (dim, m)"
    return [(int(a), int(b)) for a, b in out]


def kmeans_assign(rows, centroids, metric, sel=None, nthreads=1):
    rows, centroids = _c(rows), _c(centroids)
    n, dim = rows.shape
    lo, hi = sel if sel is not None else (0, dim)
    assert centroids.shape[1] == hi - lo
    out = np.zeros(n, np.uint32)
    lib().orc_kmeans_assign(_p(rows), n, dim, _dt(rows), _METRIC[metric], _p(centroids),
                            centroids.shape[0], lo, hi, _p(out), nthreads)
    return out


def kmeans_lloyd(rows, init_centroids, metric, max_iter, tol, sel=None):
    rows = _c(rows)
    cent = np.array(init_centroids, dtype=rows.dtype, order="C", copy=True)
    n, dim = rows.shape
    lo, hi = sel if sel is not None else (0, dim)
    iters = lib().orc_kmeans_lloyd(_p(rows), n, dim, _dt(rows), _METRIC[metric], _p(cent),
                                   cent.shape[0], lo, hi, max_iter, tol)
    return cent, iters


def kmeans_pp_init(rows, k, metric, seed, sel=None):
    rows = _c(rows)
    n, dim = rows.shape
    lo, hi = sel if sel is not None else (0, dim)
    cent = np.zeros((k, hi - lo), rows.dtype)
    rc = lib().orc_kmeans_pp_init(_p(rows), n, dim, _dt(rows), _METRIC[metric], k, lo, hi, seed, _p(cent))
    assert rc == 0
    return cent


def kmeans_pp_weights(rows, c, metric, w, sel=None, nthreads=1):
    """The k-means++ weight update (k_means.rs:75-77): returns min(w, d(c, rows[:, lo:hi])) as a new f32 array."""
    rows, c = _c(rows), _c(c)
    n, dim = rows.shape
    lo, hi = sel if sel is not None else (0, dim)
    assert c.dtype == rows.dtype and c.size == hi - lo
    out = np.array(w, dtype=np.float32, order="C", copy=True)
    assert out.shape == (n,)
    rc = lib().orc_kmeans_pp_weights(_p(rows), n, dim, _dt(rows), _METRIC[metric], _p(c), lo, hi, _p(out), nthreads)
    assert rc == 0, "kmeans_pp_weights: invalid selected range"
    return out


def find_n_nearest(v, centroids, n_probes, metric):
    v, centroids = _c(v), _c(centroids)
    out = np.zeros(min(n_probes, centroids.shape[0]), np.uint64)
    c = lib().orc_find_n_nearest(_p(v), _p(centroids), centroids.shape[0], centroids.shape[1],
                                 _dt(v), _METRIC[metric], n_probes, _p(out))
    return out[:c]


def pq_encode(rows, codebooks, m, n_bits, metric, nthreads=1):
    rows, codebooks = _c(rows), _c(codebooks)
    n, dim = rows.shape
    enc = (m + 1) // 2 if n_bits == 4 else m
    codes = np.zeros((n, enc), np.uint8)
    rc = lib().orc_pq_encode(_p(rows), n, dim, _dt(rows), _METRIC[metric], _p(codebooks), m, n_bits,
                             _p(codes), nthreads)
    assert rc == 0
    return codes


def pq_lookup(q, codebooks, m, n_bits, metric):
    q, codebooks = _c(q), _c(codebooks)
    lut = np.zeros(m * (1 << n_bits), np.float32)
    qc = np.zeros(1, np.float32)
    lib().orc_pq_lookup(_p(q), q.size, _dt(q), _METRIC[metric], _p(codebooks), m, n_bits, _p(lut), _p(qc))
    return lut, float(qc[0])


def pq_dist_cache(dim, codebooks, m, n_bits, metric):
    codebooks = _c(codebooks)
    out = np.zeros(m * (1 << n_bits), np.float32)
    lib().orc_pq_dist_cache(dim, _dt(codebooks), _METRIC[metric], _p(codebooks), m, n_bits, _p(out))
    return out


def pq_adc(codes, m, n_bits, metric, lut, dist_cache_, qcache):
    codes, lut, dist_cache_ = _c(codes), _c(lut, np.float32), _c(dist_cache_, np.float32)
    out = np.zeros(codes.shape[0], np.float32)
    L = lib()
    enc = codes.shape[1]
    base = codes.ctypes.data
    for i in range(codes.shape[0]):
        out[i] = L.orc_pq_adc(C.c_void_p(base + i * enc), m, n_bits, _METRIC[metric], _p(lut),
                              _p(dist_cache_), qcache)
    return out


def flat_adc_topk(codes, m, n_bits, metric, lut, dist_cache_, qcache, kk):
    codes, lut, dist_cache_ = _c(codes), _c(lut, np.float32), _c(dist_cache_, np.float32)
    ids = np.zeros(kk, np.uint64)
    dd = np.zeros(kk, np.float32)
    cnt = np.zeros(1, np.uint32)
    lib().orc_flat_adc_topk(codes.shape[0], _METRIC[metric], _p(codes), m, n_bits, _p(lut),
                            _p(dist_cache_), qcache, kk, _p(ids), _p(dd), _p(cnt))
    return ids[:cnt[0]], dd[:cnt[0]]


def flat_knn_pq(base, codes, codebooks, m, n_bits, queries, k, ef, metric, nthreads=1):
    base, codes, codebooks, queries = _c(base), _c(codes), _c(codebooks), _c(queries)
    n, dim = base.shape
    nq = queries.shape[0]
    ids = np.zeros((nq, k), np.uint64)
    dd = np.zeros((nq, k), np.float32)
    cnt = np.zeros(nq, np.uint32)
    rc = lib().orc_flat_knn_pq(_p(base), n, dim, _dt(base), _METRIC[metric], _p(codes), _p(codebooks),
                               m, n_bits, _p(queries), nq, k, ef, _p(ids), _p(dd), _p(cnt), nthreads)
    assert rc == 0
    return ids, dd, cnt


def ivf_lists(assign, nlist):
    assign = _c(assign, np.uint32)
    offsets = np.zeros(nlist + 1, np.uint64)
    members = np.zeros(assign.size, np.uint64)
    rc = lib().orc_ivf_lists(_p(assign), assign.size, nlist, _p(offsets), _p(members))
    assert rc == 0
    return offsets, members


def ivf_knn(base, centroids, offsets, members, queries, k, n_probes, metric, nthreads=1):
    base, centroids, queries = _c(base), _c(centroids), _c(queries)
    offsets, members = _c(offsets, np.uint64), _c(members, np.uint64)
    n, dim = base.shape
    nq = queries.shape[0]
    ids = np.zeros((nq, k), np.uint64)
    dd = np.zeros((nq, k), np.float32)
    cnt = np.zeros(nq, np.uint32)
    rc = lib().orc_ivf_knn(_p(base), n, dim, _dt(base), _METRIC[metric], _p(centroids),
                           centroids.shape[0], _p(offsets), _p(members), _p(queries), nq, k, n_probes,
                           _p(ids), _p(dd), _p(cnt), nthreads)
    assert rc == 0, "ivf_knn: n_probes must be > 0"
    return ids, dd, cnt


def gather_dist(base, row_cache, query, query_cache, cand, metric):
    base, query = _c(base), _c(query)
    row_cache, cand = _c(row_cache, np.float32), _c(cand, np.uint64)
    out = np.zeros(cand.size, np.float32)
    lib().orc_gather_dist(_p(base), base.shape[1], _dt(base), _METRIC[metric], _p(row_cache), _p(query),
                          query_cache, _p(cand), cand.size, _p(out))
    return out


def recall(gnd, pred):
    gnd, pred = _c(gnd, np.uint64), _c(pred, np.uint64)
    return lib().orc_recall(_p(gnd), gnd.size, _p(pred), pred.size)


_KNN_ARGS = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p,
             C.c_int, C.c_void_p]
_KNN_PQ_ARGS = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_void_p, C.c_void_p, C.c_size_t,
                C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]


class HnswOracle:
    """Single-thread restatement of HNSWIndex (sequential add of every row, knn_with_ef); recall yardstick.

    Tie events: an add to a full result set with a distance equal to its last entry's. The reference keeps the older
    entry whatever the ids, a selection of the smallest (distance, id) keys may keep the newer one; on data where every
    distance is exact that is the only way two correct walks over the same graph can differ. `build_ties` counts them
    over a build, `knn(..., ties=True)` per query."""

    def __init__(self, base, metric, m, ef_construction, levels):
        self.base = _c(base)
        self.dt = _dt(self.base)
        levels = _c(levels, np.uint32)
        self.levels = levels
        f = lib().orc_hnsw_build
        f.restype = C.c_void_p
        f.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_void_p]
        lib().orc_hnsw_links0.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        lib().orc_hnsw_free.argtypes = [C.c_void_p, C.c_int]
        lib().orc_hnsw_free.restype = None
        self.h = C.c_void_p(f(_p(self.base), C.c_size_t(self.base.shape[0]), C.c_size_t(self.base.shape[1]),
                                   self.dt, _METRIC[metric], C.c_size_t(m), C.c_size_t(ef_construction), _p(levels)))
        self.m = m

    @classmethod
    def from_graph(cls, base, metric, m, ef_construction, levels, links0, len0, ulinks, ulen, enter_point, enter_level):
        """The CPU search over a graph built elsewhere (e.g. by the GPU build): layouts of vdb_hnsw_links0 / _upper."""
        self = cls.__new__(cls)
        self.base = _c(base)
        self.dt = _dt(self.base)
        self.levels = _c(levels, np.uint32)
        self.m = m
        self._keep = (_c(links0, np.uint32), _c(len0, np.uint32), _c(ulinks, np.uint32), _c(ulen, np.uint32))
        f = lib().orc_hnsw_from_graph
        f.restype = C.c_void_p
        f.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_void_p, C.c_void_p,
                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_long, C.c_long]
        lib().orc_hnsw_free.argtypes = [C.c_void_p, C.c_int]
        lib().orc_hnsw_free.restype = None
        ul = self._keep[2] if self._keep[2].size else np.zeros(1, np.uint32)
        un = self._keep[3] if self._keep[3].size else np.zeros(1, np.uint32)
        self.h = C.c_void_p(f(_p(self.base), self.base.shape[0], self.base.shape[1], self.dt, _METRIC[metric], m,
                              ef_construction, _p(self.levels), _p(self._keep[0]), _p(self._keep[1]), _p(ul), _p(un),
                              int(enter_point), int(enter_level)))
        return self

    @classmethod
    def batched(cls, base, metric, m, ef_construction, levels, max_batch, n0=0):
        """The device build's batch pipeline (orc_hnsw_build_batched): a build of rows [0, n0), then an append of the
        rest onto it (n0 = 0: one build of every row)."""
        self = cls.__new__(cls)
        self.base = _c(base)
        self.dt = _dt(self.base)
        self.levels = _c(levels, np.uint32)
        self.m = m
        f = lib().orc_hnsw_build_batched
        f.restype = C.c_void_p
        f.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_void_p, C.c_size_t,
                      C.c_size_t]
        h = f(_p(self.base), self.base.shape[0], self.base.shape[1], self.dt, _METRIC[metric], m, ef_construction,
              _p(self.levels), max_batch, n0)
        assert h, "orc_hnsw_build_batched: max_batch must be positive and n0 <= n"
        self.h = C.c_void_p(h)
        return self

    @property
    def build_ties(self):
        f = lib().orc_hnsw_build_ties
        f.restype = C.c_uint64
        f.argtypes = [C.c_void_p, C.c_int]
        return int(f(self.h, self.dt))

    @property
    def enter_point(self):
        """(enter point, enter level), like HNSWIndex.enter_point"""
        f = lib().orc_hnsw_enter
        f.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        ep, el = C.c_long(-1), C.c_long(-1)
        f(self.h, self.dt, C.byref(ep), C.byref(el))
        return int(ep.value), int(el.value)

    def knn(self, queries, k, ef, nthreads=1, ties=False):
        """(ids, dist, counts), and with ties=True the tie events of every query's walk as a fourth array"""
        q = _c(queries)
        nq = q.shape[0]
        ids = np.zeros((nq, k), np.uint64)
        dd = np.zeros((nq, k), np.float32)
        cnt = np.zeros(nq, np.uint32)
        tie = np.zeros(max(nq, 1), np.uint32)
        f = lib().orc_hnsw_knn
        f.argtypes = _KNN_ARGS
        f(self.h, self.dt, _p(q), nq, k, ef, _p(ids), _p(dd), _p(cnt), nthreads, _p(tie))
        return (ids, dd, cnt, tie[:nq]) if ties else (ids, dd, cnt)

    def knn_pq(self, queries, k, ef, codes, codebooks, m, n_bits, nthreads=1, ties=False):
        """(ids, dist, counts), and with ties=True the tie events of every query's walk and resort"""
        q, codes, codebooks = _c(queries), _c(codes, np.uint8), _c(codebooks)
        nq = q.shape[0]
        ids = np.zeros((nq, k), np.uint64)
        dd = np.zeros((nq, k), np.float32)
        cnt = np.zeros(nq, np.uint32)
        tie = np.zeros(max(nq, 1), np.uint32)
        f = lib().orc_hnsw_knn_pq
        f.argtypes = _KNN_PQ_ARGS
        f(self.h, self.dt, _p(q), nq, k, ef, _p(codes), _p(codebooks), m, n_bits, _p(ids), _p(dd), _p(cnt), nthreads,
          _p(tie))
        return (ids, dd, cnt, tie[:nq]) if ties else (ids, dd, cnt)

    def links0(self):
        n = self.base.shape[0]
        links = np.zeros((n, 2 * self.m), np.uint32)
        lens = np.zeros(n, np.uint32)
        lib().orc_hnsw_links0(self.h, self.dt, _p(links), _p(lens))
        return links, lens

    def upper(self):
        slots = int(self.levels.sum())
        ul = np.zeros(max(slots, 1) * self.m, np.uint32)
        un = np.zeros(max(slots, 1), np.uint32)
        f = lib().orc_hnsw_upper
        f.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        f(self.h, self.dt, _p(ul), _p(un))
        return ul[:slots * self.m], un[:slots]

    def __del__(self):
        try:
            f = lib().orc_hnsw_free
            f.restype = None
            f(self.h, self.dt)
        except Exception:
            pass
