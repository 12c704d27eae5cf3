"""Host-side mirror of the reference's index_algorithm surface for the GPU path.

Names follow the reference: FlatIndex.from_vec_set / knn (src/index_algorithm/flat_index.rs:48-70),
CandidatePair (src/index_algorithm/candidate_pair.rs:10-40). `knn_batch` is the additive batch entry
(the reference is single-query; examples/bench.rs:414-418 batches with rayon instead).
"""
import ctypes as C
from typing import List, NamedTuple

import numpy as np

from . import _lib as L


class CandidatePair(NamedTuple):
    """(index, distance) as returned by IndexKNN::knn; ordered by (distance, index)."""
    index: int
    distance: float


def _as_rows(a, dtype=None):
    a = np.asarray(a)
    if dtype is not None and a.dtype != dtype:
        raise TypeError(f"expected {dtype}, got {a.dtype}")
    if a.ndim == 1:
        a = a.reshape(1, -1)
    return np.ascontiguousarray(a)


def init_devices(devices):
    """vdb_init: the CUDA devices of this process. With two or more, DeviceVecSet(rows) row-shards the set over them
    and every FlatIndex.knn / knn_batch on it is ONE C call that runs on all of them (peer-memory merge). A device may
    be listed several times (several shards on one GPU). [] returns to single-device mode."""
    arr = (C.c_int * max(1, len(devices)))(*devices)
    L.check(L.lib().vdb_init(arr, len(devices)))


class DeviceVecSet:
    """Device mirror of VecSet<T> (reference src/vec_set.rs:15-30) — one row shard in HBM, or, after
    init_devices([...]) with several devices, the whole set row-sharded over them."""

    def __init__(self, rows, dist="l2sqr", id_base=0):
        rows = np.ascontiguousarray(rows)
        if rows.ndim != 2:
            raise ValueError("rows must be [n, dim]")
        self.dtype = rows.dtype
        self.dim = int(rows.shape[1])
        self.metric = L.metric_code(dist)
        self.id_base = int(id_base)
        self._h = C.c_void_p()
        L.check(L.lib().vdb_dataset_create(L.ptr(rows), rows.shape[0], self.dim, L.dtype_code(rows),
                                           self.metric, self.id_base, C.byref(self._h)))
        self._keepalive = None

    @classmethod
    def from_device(cls, d_ptr, n, dim, pitch, dtype, dist="l2sqr", id_base=0, keepalive=None):
        """Adopts rows already resident in HBM (e.g. a torch tensor's data_ptr())."""
        self = cls.__new__(cls)
        self.dtype = np.dtype(dtype)
        self.dim = int(dim)
        self.metric = L.metric_code(dist)
        self.id_base = int(id_base)
        self._h = C.c_void_p()
        code = L.F32 if self.dtype == np.float32 else L.U8
        L.check(L.lib().vdb_dataset_create_dev(C.c_void_p(int(d_ptr)), n, dim, pitch, code, self.metric,
                                               self.id_base, C.byref(self._h)))
        self._keepalive = keepalive
        return self

    @classmethod
    def from_device_shards(cls, d_ptrs, counts, devices, dim, pitch, dtype, dist="l2sqr", id_base=0, keepalive=None):
        """Row-sharded set over rows already resident on the shards' devices (shard s: counts[s] rows at d_ptrs[s] on
        devices[s]); enables peer access between the devices."""
        self = cls.__new__(cls)
        self.dtype = np.dtype(dtype)
        self.dim = int(dim)
        self.metric = L.metric_code(dist)
        self.id_base = int(id_base)
        self._h = C.c_void_p()
        g = len(d_ptrs)
        code = L.F32 if self.dtype == np.float32 else L.U8
        L.check(L.lib().vdb_dataset_create_sharded_dev((C.c_void_p * g)(*[int(p) for p in d_ptrs]),
                                                       (C.c_uint64 * g)(*[int(c) for c in counts]),
                                                       (C.c_int * g)(*[int(d) for d in devices]), g, dim, pitch, code,
                                                       self.metric, self.id_base, C.byref(self._h)))
        self._keepalive = keepalive
        return self

    def shards(self):
        """[(device, row_lo, row_hi)] of a row-sharded set, [] otherwise."""
        n = C.c_uint32()
        L.check(L.lib().vdb_dataset_shards(self._h, C.byref(n)))
        out = []
        for s in range(n.value):
            dev, lo, hi = C.c_int(), C.c_uint64(), C.c_uint64()
            L.check(L.lib().vdb_dataset_shard(self._h, s, None, C.byref(dev), C.byref(lo), C.byref(hi)))
            out.append((dev.value, int(lo.value), int(hi.value)))
        return out

    def set_flat_path(self, path):
        """Flat implementation for THIS handle: "auto", "scan" (K1), "tensor" (K2) or None (process default)."""
        code = {None: -1, "auto": 0, "scan": 1, "tensor": 2}[path]
        L.check(L.lib().vdb_dataset_set_flat_path(self._h, code))

    def __len__(self):
        n = C.c_uint64()
        L.check(L.lib().vdb_dataset_len(self._h, C.byref(n)))
        return int(n.value)

    def push(self, rows):
        """VecSet::push (src/vec_set.rs:113-118), batched."""
        rows = _as_rows(rows, self.dtype)
        if rows.shape[1] != self.dim:
            raise ValueError("The dimension of the vector doesn't match.")
        L.check(L.lib().vdb_dataset_append(self._h, L.ptr(rows), rows.shape[0]))

    def swap_remove(self, idx):
        """VecSet::swap_remove (src/vec_set.rs:131-137)."""
        L.check(L.lib().vdb_dataset_swap_remove(self._h, int(idx)))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            L.lib().vdb_dataset_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _pairs(ids, dist, counts):
    out = []
    for q in range(ids.shape[0]):
        c = int(counts[q])
        out.append([CandidatePair(int(ids[q, j]), float(dist[q, j])) for j in range(c)])
    return out


class FlatIndex:
    """FlatIndex<T> (reference src/index_algorithm/flat_index.rs:17-57) backed by the GPU scan."""

    def __init__(self, vec_set: DeviceVecSet):
        self.vec_set = vec_set

    @classmethod
    def from_vec_set(cls, vec_set, dist="l2sqr", config=None, rng=None):
        """IndexFromVecSet::from_vec_set (flat_index.rs:59-70); `config`/`rng` are unused as there."""
        if not isinstance(vec_set, DeviceVecSet):
            vec_set = DeviceVecSet(vec_set, dist)
        return cls(vec_set)

    def __len__(self):
        return len(self.vec_set)

    def dim(self):
        return self.vec_set.dim

    def knn_batch(self, queries, k, out=None):
        """Returns (ids [nq,k] u64, dist [nq,k] f32, counts [nq] u32). `out` = caller-owned result arrays of those
        shapes / dtypes to reuse across calls (e.g. page-locked memory), as a Rust caller reuses its Vecs."""
        vs = self.vec_set
        q = _as_rows(queries, vs.dtype)
        if q.shape[1] != vs.dim:
            raise ValueError("The dimension of the query doesn't match.")
        nq = q.shape[0]
        if out is not None:
            ids, dist, counts = out
            if not (ids.shape == (nq, k) and ids.dtype == np.uint64 and ids.flags.c_contiguous and
                    dist.shape == (nq, k) and dist.dtype == np.float32 and dist.flags.c_contiguous and
                    counts.shape == (nq,) and counts.dtype == np.uint32 and counts.flags.c_contiguous):
                raise ValueError("out must be C-contiguous (u64 [nq,k], f32 [nq,k], u32 [nq]) arrays")
        else:
            ids = np.full((nq, k), np.iinfo(np.uint64).max, np.uint64)
            dist = np.full((nq, k), np.nan, np.float32)
            counts = np.zeros(nq, np.uint32)
        L.check(L.lib().vdb_flat_knn(vs._h, L.ptr(q), nq, k, L.ptr(ids), L.ptr(dist), L.ptr(counts)))
        return ids, dist, counts

    def knn(self, query, k) -> List[CandidatePair]:
        """IndexKNN::knn (flat_index.rs:48-57)."""
        ids, dist, counts = self.knn_batch(np.asarray(query).reshape(1, -1), k)
        return _pairs(ids, dist, counts)[0]

    def knn_batch_sharded_dev(self, d_queries, nq, k, d_ids, d_dist, d_counts):
        """Device-resident search on a row-sharded set (vdb_flat_knn_sharded_dev): d_queries[s] = pointer of the whole
        batch on shard s's device; shard s receives the results of queries [s * per, (s + 1) * per), per = ceil(nq / G),
        in d_ids[s] / d_dist[s] / d_counts[s]. Pointers are raw integers. Synchronous."""
        g = len(d_queries)
        arr = lambda ps: (C.c_void_p * g)(*[int(p) for p in ps])  # noqa: E731
        L.check(L.lib().vdb_flat_knn_sharded_dev(self.vec_set._h, arr(d_queries), nq, k, arr(d_ids), arr(d_dist),
                                                 arr(d_counts)))


def calc_dist(a, b, dist="cosine"):
    """calc_dist(a, b, dist="cosine") of the pyo3 layer (reference src/pyo3/mod.rs:43-48)."""
    a = np.ascontiguousarray(a, dtype=np.float32).reshape(-1)
    b = np.ascontiguousarray(b, dtype=np.float32).reshape(-1)
    if a.size != b.size:
        raise ValueError("The dimension of the vectors doesn't match.")
    out = np.zeros(1, np.float32)
    L.check(L.lib().vdb_calc_dist(L.ptr(a), L.ptr(b), 1, a.size, L.F32, L.metric_code(dist), L.ptr(out)))
    return float(out[0])


# ---------------------------------------------------------------------------------------------------
# distance primitives
# ---------------------------------------------------------------------------------------------------
def calc_dist_batch(a, b, dist="l2sqr"):
    """DistanceAdapter<[T],[T]>::distance for row pairs (a[i], b[i]); dist may also be "dot"."""
    a, b = _as_rows(a), _as_rows(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        raise ValueError("The dimension of the vectors doesn't match.")
    code = L.DOT if (isinstance(dist, str) and dist.lower() == "dot") else L.metric_code(dist)
    out = np.zeros(a.shape[0], np.float32)
    L.check(L.lib().vdb_calc_dist(L.ptr(a), L.ptr(b), a.shape[0], a.shape[1], L.dtype_code(a), code, L.ptr(out)))
    return out


def dist_cache(vec_set: DeviceVecSet):
    """DistanceAlgorithm::dist_cache for every row (distance/mod.rs:31-36)."""
    out = np.zeros(len(vec_set), np.float32)
    L.check(L.lib().vdb_row_cache(vec_set._h, L.ptr(out)))
    return out


def gather_dist(vec_set: DeviceVecSet, queries, cand_lists):
    """Batched cached-form distances for HNSW frontier expansion (hnsw_index.rs:351-358).
    cand_lists[j] = local row ids to compare with queries[j]. Returns a list of f32 arrays."""
    q = _as_rows(queries, vec_set.dtype)
    off = np.zeros(len(cand_lists) + 1, np.uint64)
    off[1:] = np.cumsum([len(c) for c in cand_lists])
    ids = (np.concatenate([np.asarray(c, np.uint32) for c in cand_lists]) if len(cand_lists) and off[-1]
           else np.zeros(0, np.uint32))
    out = np.zeros(int(off[-1]), np.float32)
    L.check(L.lib().vdb_gather_dist(vec_set._h, L.ptr(q), q.shape[0], L.ptr(ids) if ids.size else None,
                                    L.ptr(off), L.ptr(out) if out.size else None))
    return [out[int(off[j]):int(off[j + 1])] for j in range(len(cand_lists))]


# ---------------------------------------------------------------------------------------------------
# k-means (reference src/distance/k_means.rs)
# ---------------------------------------------------------------------------------------------------
class KMeansConfig(NamedTuple):
    """KMeansConfig (k_means.rs:15-31)."""
    k: int
    max_iter: int = 20
    tol: float = 1e-6
    dist: str = "l2sqr"
    selected: tuple = None


def _as_device_rows(rows, dist):
    """Training rows as a DeviceVecSet (uploaded once; PQ trains one k-means per group on the same sample)."""
    if isinstance(rows, DeviceVecSet):
        return rows
    return DeviceVecSet(np.ascontiguousarray(rows), dist)


def sample_indices(rng, n, k):
    """Row indices of VecSet::random_sample (vec_set.rs:154-163): the first k entries of the shuffled index vector. A
    `rand_compat.StdRng` follows the reference's Fisher-Yates draws, a numpy Generator its own permutation."""
    from .rand_compat import StdRng
    if isinstance(rng, StdRng):
        return rng.shuffle(n)[:k]
    return rng.permutation(n)[:k]


def k_means_init_reference_stream(rows_host, config: KMeansConfig, rng):
    """k-means++ (k_means.rs:61-87) under the reference's OWN random stream (`rand_compat.StdRng`: rand 0.8.5 restated,
    parity with the crate unpinned - see that module): gen_range for the first pick, per round the f32 WeightedIndex over
    the weights the GPU updates (`vdb_kmeans_pp_weights`: w[i] = min(w[i], d(c, v_i)) with the reference's sequential f32
    distance) and the eagerly drawn fallback. Rows stay on the host (the weights call stages them)."""
    from .rand_compat import k_means_init_indices
    rows = np.ascontiguousarray(rows_host)
    n, dim = rows.shape
    lo, hi = config.selected if config.selected is not None else (0, dim)
    w = np.full(n, np.inf, np.float32)

    def update(idx):
        c = np.ascontiguousarray(rows[idx, lo:hi])
        L.check(L.lib().vdb_kmeans_pp_weights(L.ptr(rows), n, dim, L.dtype_code(rows), L.metric_code(config.dist), L.ptr(c),
                                              lo, hi, L.ptr(w)))
        return w

    chosen = k_means_init_indices(update, n, config.k, rng)
    return np.ascontiguousarray(rows[chosen, lo:hi])


def k_means_init(rows, config: KMeansConfig, rng):
    """k-means++ (k_means.rs:61-87). The draws consume the CALLER's rng: with a numpy Generator 2k-1 uniforms drive the
    first pick, the weighted picks and the eagerly drawn fallbacks and everything runs on the GPU over device-resident
    rows; with a `rand_compat.StdRng` the reference's draw sequence is followed (k_means_init_reference_stream)."""
    from .rand_compat import StdRng
    if isinstance(rng, StdRng):
        if isinstance(rows, DeviceVecSet):
            raise TypeError("the reference-stream k-means++ needs the training rows on the host (pass the numpy array)")
        return k_means_init_reference_stream(rows, config, rng)
    vs = _as_device_rows(rows, config.dist)
    lo, hi = config.selected if config.selected is not None else (0, vs.dim)
    u = np.ascontiguousarray(rng.random(2 * config.k - 1), dtype=np.float64)
    cent = np.zeros((config.k, hi - lo), vs.dtype)
    L.check(L.lib().vdb_kmeans_pp_init_ds(vs._h, config.k, lo, hi, L.ptr(u), L.ptr(cent)))
    return cent


class KMeans:
    """KMeans<T> (k_means.rs:34-37, 95-191)."""

    def __init__(self, config: KMeansConfig, centroids):
        self.config = config
        self.centroids = np.ascontiguousarray(centroids)

    @classmethod
    def from_vec_set(cls, rows, config: KMeansConfig, rng=None, init_centroids=None):
        """KMeans::from_vec_set (k_means.rs:95-162). `rows` may be a host array or a DeviceVecSet."""
        if config.k <= 0:
            raise ValueError("The number of clusters should be greater than 0.")
        from .rand_compat import StdRng
        if init_centroids is None and isinstance(rng, StdRng):
            init_centroids = k_means_init(rows, config, rng)   # the reference's stream: host rows (see k_means_init)
        vs = _as_device_rows(rows, config.dist)
        dim = vs.dim
        lo, hi = config.selected if config.selected is not None else (0, dim)
        if hi > dim:
            raise ValueError("The selected range should be in the range [0, vec_set.dim())")
        if init_centroids is None:
            init_centroids = k_means_init(vs, config, rng if rng is not None else np.random.default_rng())
        cent = np.array(init_centroids, dtype=vs.dtype, order="C", copy=True)
        iters = C.c_uint32(0)
        L.check(L.lib().vdb_kmeans_train_ds(vs._h, L.ptr(cent), config.k, lo, hi, config.max_iter, config.tol,
                                            C.byref(iters)))
        self = cls(config, cent)
        self.iterations = int(iters.value)
        return self

    def find_nearest_batch(self, rows):
        rows = _as_rows(rows, self.centroids.dtype)
        n, dim = rows.shape
        lo, hi = self.config.selected if self.config.selected is not None else (0, dim)
        out = np.zeros(n, np.uint32)
        L.check(L.lib().vdb_kmeans_assign(L.ptr(rows), n, dim, L.dtype_code(rows), L.metric_code(self.config.dist),
                                          L.ptr(self.centroids), self.centroids.shape[0], lo, hi, L.ptr(out)))
        return out

    def find_nearest(self, v):
        """KMeans::find_nearest (k_means.rs:166-170)."""
        return int(self.find_nearest_batch(np.asarray(v).reshape(1, -1))[0])


# ---------------------------------------------------------------------------------------------------
# PQ (reference src/distance/pq_table.rs)
# ---------------------------------------------------------------------------------------------------
def pq_groups(dim, m):
    """pq_groups (pq_table.rs:38-53)."""
    out = np.zeros((max(m, 1), 2), np.uint32)
    L.check(L.lib().vdb_pq_groups(dim, m, L.ptr(out)))
    return [(int(a), int(b)) for a, b in out[:m]]


class PQConfig(NamedTuple):
    """PQConfig (pq_table.rs:19-34)."""
    n_bits: int
    m: int
    dist: str = "l2sqr"
    k_means_size: int = None
    k_means_max_iter: int = 20
    k_means_tol: float = 1e-6


def train_codebooks(train_dev: DeviceVecSet, config: "PQConfig", rng=None, init_codebooks=None):
    """The m per-group k-means of PQTable::from_vec_set (pq_table.rs:154-172) on a device-resident sample. All groups
    are trained by one launch (vdb_pq_train_ds); the per-group path remains for shapes that do not fit one CTA."""
    rng = rng if rng is not None else np.random.default_rng()
    k, dim = 1 << config.n_bits, train_dev.dim
    total = sum((hi - lo) * k for lo, hi in pq_groups(dim, config.m))
    books = np.zeros(total, train_dev.dtype)
    iters = np.zeros(config.m, np.uint32)
    uni = None if init_codebooks is not None else np.ascontiguousarray(rng.random((config.m, 2 * k - 1)))
    init = None if init_codebooks is None else np.ascontiguousarray(init_codebooks, dtype=train_dev.dtype)
    rc = L.lib().vdb_pq_train_ds(train_dev._h, config.m, config.n_bits, config.k_means_max_iter, config.k_means_tol,
                                 L.ptr(uni), L.ptr(init), L.ptr(books), L.ptr(iters))
    if rc == L.EUNSUPPORTED:
        parts, o = [], 0
        for lo, hi in pq_groups(dim, config.m):
            ini = None if init is None else init[o:o + k * (hi - lo)].reshape(k, hi - lo)
            o += k * (hi - lo)
            km = KMeans.from_vec_set(train_dev, KMeansConfig(k, config.k_means_max_iter, config.k_means_tol, config.dist,
                                                             (lo, hi)), rng, ini)
            parts.append(km.centroids.reshape(-1))
        return np.concatenate(parts)
    L.check(rc)
    train_codebooks.last_iterations = iters
    return books


class PQTable:
    """PQTable<T> (pq_table.rs:116-137): codebooks + codes, device resident."""

    def __init__(self, vec_set: DeviceVecSet, config: PQConfig, codebooks, codes=None):
        if config.n_bits not in (4, 8):
            raise ValueError("n_bits must be 4 or 8 in PQTable.")
        self.config = config
        self.vec_set = vec_set
        self.dim = vec_set.dim
        self.k = 1 << config.n_bits
        self.encoded_dim = (config.m + 1) // 2 if config.n_bits == 4 else config.m
        self.codebooks = np.ascontiguousarray(codebooks, dtype=vec_set.dtype).reshape(-1)
        self._h = C.c_void_p()
        n = len(vec_set)
        if codes is None:
            self.encoded_vec_set = np.zeros((n, self.encoded_dim), np.uint8)
            L.check(L.lib().vdb_pq_create(vec_set._h, L.ptr(self.codebooks), config.m, config.n_bits,
                                          L.ptr(self.encoded_vec_set), C.byref(self._h)))
        else:
            self.encoded_vec_set = np.ascontiguousarray(codes, np.uint8)
            L.check(L.lib().vdb_pq_create_from_codes(vec_set._h, L.ptr(self.codebooks), config.m, config.n_bits,
                                                     L.ptr(self.encoded_vec_set), C.byref(self._h)))

    @classmethod
    def from_vec_set(cls, vec_set, rows_host, config: PQConfig, rng=None):
        """PQTable::from_vec_set (pq_table.rs:141-191): sample, per-group k-means, encode."""
        rng = rng if rng is not None else np.random.default_rng()
        rows_host = np.ascontiguousarray(rows_host)
        train = rows_host
        if config.k_means_size is not None:
            perm = sample_indices(rng, len(rows_host), config.k_means_size)  # VecSet::random_sample (vec_set.rs:154-163)
            train = np.ascontiguousarray(rows_host[perm])
        train_dev = DeviceVecSet(train, config.dist)  # the sample is uploaded once for all m groups
        try:
            from .rand_compat import StdRng
            init = None
            if isinstance(rng, StdRng):
                # the reference trains the groups one after the other on one stream (pq_table.rs:154-172); only the
                # k-means++ of each group draws, so the initial centroids are fixed here in group order and Lloyd runs
                # for all groups at once (bit-identical to the per-group runs given the same start)
                k = 1 << config.n_bits
                init = np.concatenate([
                    k_means_init(train, KMeansConfig(k, config.k_means_max_iter, config.k_means_tol, config.dist, (lo, hi)),
                                 rng).reshape(-1) for lo, hi in pq_groups(train.shape[1], config.m)])
            books = train_codebooks(train_dev, config, rng, init)
        finally:
            train_dev.close()
        return cls(vec_set, config, books)

    def create_lookup(self, queries):
        """PQTable::create_lookup (pq_table.rs:195-224) -> (lookup [nq, m*k], dist_cache [nq])."""
        q = _as_rows(queries, self.vec_set.dtype)
        lut = np.zeros((q.shape[0], self.config.m * self.k), np.float32)
        qc = np.zeros(q.shape[0], np.float32)
        L.check(L.lib().vdb_pq_lut(self._h, L.ptr(q), q.shape[0], L.ptr(lut), L.ptr(qc)))
        return lut, qc

    def adc_distances(self, queries):
        """ADC distance of every code (pq_table.rs:239-301) -> [nq, n]."""
        q = _as_rows(queries, self.vec_set.dtype)
        out = np.zeros((q.shape[0], len(self.vec_set)), np.float32)
        L.check(L.lib().vdb_pq_adc_all(self._h, L.ptr(q), q.shape[0], L.ptr(out)))
        return out

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            L.lib().vdb_pq_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _knn_pq_batch(self, queries, k, ef, pq_table):
    vs = self.vec_set
    q = _as_rows(queries, vs.dtype)
    if q.shape[1] != vs.dim:
        raise ValueError("The dimension of the query doesn't match.")
    if L.metric_code(pq_table.config.dist) != vs.metric:
        raise ValueError("Distance algorithm mismatch.")
    nq = q.shape[0]
    ids = np.full((nq, k), np.iinfo(np.uint64).max, np.uint64)
    dist = np.full((nq, k), np.nan, np.float32)
    counts = np.zeros(nq, np.uint32)
    L.check(L.lib().vdb_pq_knn(vs._h, pq_table._h, L.ptr(q), nq, k, ef, L.ptr(ids), L.ptr(dist), L.ptr(counts)))
    return ids, dist, counts


def _knn_pq(self, query, k, ef, pq_table):
    """IndexPQ::knn_pq (flat_index.rs:84-104)."""
    return _pairs(*_knn_pq_batch(self, np.asarray(query).reshape(1, -1), k, ef, pq_table))[0]


FlatIndex.knn_pq_batch = _knn_pq_batch
FlatIndex.knn_pq = _knn_pq


# ---------------------------------------------------------------------------------------------------
# IVF (reference src/index_algorithm/ivf_index.rs)
# ---------------------------------------------------------------------------------------------------
class IVFConfig(NamedTuple):
    """IVFConfig (ivf_index.rs:20-31)."""
    k: int
    k_means_size: int = None
    k_means_max_iter: int = 20
    k_means_tol: float = 1e-6


class IVFIndex:
    """IVFIndex<T> (ivf_index.rs:34-47)."""

    def __init__(self, vec_set: DeviceVecSet, centroids, config: IVFConfig = None):
        self.vec_set = vec_set
        self.config = config
        self.default_n_probes = 4  # ivf_index.rs:97
        self.centroids = np.ascontiguousarray(centroids, dtype=vec_set.dtype)
        self._h = C.c_void_p()
        self.assignment = np.zeros(len(vec_set), np.uint32)
        L.check(L.lib().vdb_ivf_create(vec_set._h, L.ptr(self.centroids), self.centroids.shape[0],
                                       L.ptr(self.assignment), C.byref(self._h)))

    @classmethod
    def from_vec_set(cls, vec_set, rows_host, dist, config: IVFConfig, rng=None):
        """IndexFromVecSet::from_vec_set (ivf_index.rs:67-107)."""
        rng = rng if rng is not None else np.random.default_rng()
        rows_host = np.ascontiguousarray(rows_host)
        train = rows_host
        if config.k_means_size is not None:
            train = np.ascontiguousarray(rows_host[sample_indices(rng, len(rows_host), config.k_means_size)])
        km = KMeans.from_vec_set(train, KMeansConfig(config.k, config.k_means_max_iter, config.k_means_tol, dist), rng)
        if not isinstance(vec_set, DeviceVecSet):
            vec_set = DeviceVecSet(rows_host, dist)
        return cls(vec_set, km.centroids, config)

    @property
    def clusters(self):
        off = np.zeros(self.centroids.shape[0] + 1, np.uint64)
        mem = np.zeros(len(self.vec_set), np.uint32)
        L.check(L.lib().vdb_ivf_lists(self._h, L.ptr(off), L.ptr(mem)))
        return [mem[int(off[c]):int(off[c + 1])] for c in range(self.centroids.shape[0])]

    def set_default_ef(self, n_probes):
        self.default_n_probes = n_probes

    def knn_with_ef_batch(self, queries, k, n_probes):
        vs = self.vec_set
        q = _as_rows(queries, vs.dtype)
        if q.shape[1] != vs.dim:
            raise ValueError("The dimension of the query doesn't match.")
        if n_probes <= 0:
            raise ValueError("The number of probes should be greater than 0.")
        nq = q.shape[0]
        ids = np.full((nq, k), np.iinfo(np.uint64).max, np.uint64)
        dist = np.full((nq, k), np.nan, np.float32)
        counts = np.zeros(nq, np.uint32)
        L.check(L.lib().vdb_ivf_knn(vs._h, self._h, L.ptr(q), nq, k, n_probes, L.ptr(ids), L.ptr(dist), L.ptr(counts)))
        return ids, dist, counts

    def knn_with_ef(self, query, k, n_probes):
        """IndexKNNWithEf::knn_with_ef (ivf_index.rs:143-154); ef = number of probes."""
        return _pairs(*self.knn_with_ef_batch(np.asarray(query).reshape(1, -1), k, n_probes))[0]

    def knn(self, query, k):
        return self.knn_with_ef(query, k, self.default_n_probes)

    def knn_pq_batch(self, queries, k, ef, pq_table, n_probes=None):
        """IndexPQ::knn_pq restricted to the n_probes nearest lists (default: default_n_probes): the max(ef, k) best
        codes by (ADC, id) over the rows of those lists, re-scored exactly, the k best kept. With n_probes >= nlist
        this is FlatIndex.knn_pq_batch. Returns (ids [nq,k] u64, dist [nq,k] f32, counts [nq] u32)."""
        vs = self.vec_set
        q = _as_rows(queries, vs.dtype)
        if q.shape[1] != vs.dim:
            raise ValueError("The dimension of the query doesn't match.")
        if L.metric_code(pq_table.config.dist) != vs.metric:
            raise ValueError("Distance algorithm mismatch.")
        n_probes = self.default_n_probes if n_probes is None else n_probes
        if n_probes <= 0:
            raise ValueError("The number of probes should be greater than 0.")
        nq = q.shape[0]
        ids = np.full((nq, k), np.iinfo(np.uint64).max, np.uint64)
        dist = np.full((nq, k), np.nan, np.float32)
        counts = np.zeros(nq, np.uint32)
        L.check(L.lib().vdb_ivf_knn_pq(vs._h, self._h, pq_table._h, L.ptr(q), nq, k, ef, n_probes, L.ptr(ids), L.ptr(dist),
                                       L.ptr(counts)))
        return ids, dist, counts

    def knn_pq(self, query, k, ef, pq_table):
        """IndexPQ::knn_pq with the index's default probe count (ivf_index.rs:97, set_default_ef)."""
        return _pairs(*self.knn_pq_batch(np.asarray(query).reshape(1, -1), k, ef, pq_table))[0]

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            L.lib().vdb_ivf_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---- HNSW --------------------------------------------------------------------------------------------------------
class HNSWConfig(NamedTuple):
    """HNSWConfig (hnsw_index.rs:41-71)."""
    max_elements: int = 0
    ef_construction: int = 200
    M: int = 16


def hnsw_rand_levels(n, M, rng):
    """rand_level (hnsw_index.rs:145-149) for n rows in row order: floor(-ln(u) / ln(M)), u uniform f32 in [0, 1)."""
    from .rand_compat import StdRng
    u = rng.gen_unit_f32_array(n) if isinstance(rng, StdRng) else rng.random(n, dtype=np.float32)
    u = np.maximum(u, np.float32(2.0 ** -24))  # the reference would overflow usize on u == 0
    inv_log_m = np.float32(1.0) / np.log(np.float32(M))
    return np.floor(-np.log(u) * inv_log_m).astype(np.uint32)


class HNSWIndex:
    """HNSWIndex<T> (hnsw_index.rs:99-141): the graph lives in HBM, built batch by batch on the device."""

    MAX_BATCH = 2048

    def __init__(self, vec_set: DeviceVecSet, config: HNSWConfig = HNSWConfig(), rng=None, levels=None):
        self.vec_set = vec_set
        self.config = config
        rng = rng if rng is not None else np.random.default_rng()
        n = len(vec_set)
        self.levels = (np.ascontiguousarray(levels, dtype=np.uint32) if levels is not None
                       else hnsw_rand_levels(n, config.M, rng))
        if self.levels.shape != (n,):
            raise ValueError("one level per row is required")
        self._h = C.c_void_p()
        L.check(L.lib().vdb_hnsw_build(vec_set._h, config.M, config.ef_construction, L.ptr(self.levels), self.MAX_BATCH,
                                       C.byref(self._h)))
        efc = C.c_uint32(0)
        L.check(L.lib().vdb_hnsw_info(self._h, None, None, C.byref(efc), None, None))
        self.ef_construction = int(efc.value)
        self.default_ef = self.ef_construction // 2  # hnsw_index.rs:505

    @classmethod
    def build_on_vec_set(cls, vec_set, dist="l2sqr", config: HNSWConfig = HNSWConfig(), rng=None):
        """IndexBuilder::build_on_vec_set (hnsw_index.rs:585-600)."""
        if not isinstance(vec_set, DeviceVecSet):
            vec_set = DeviceVecSet(vec_set, dist)
        return cls(vec_set, config, rng)

    from_vec_set = build_on_vec_set

    def batch_add_pushed(self, rng=None, levels=None):
        """IndexBuilder::batch_add (hnsw_index.rs:573-575) for the rows pushed to `vec_set` since the last build / add:
        they are inserted into the existing graph with the same batch pipeline as the build."""
        n_old, n = len(self.levels), len(self.vec_set)
        if n == n_old:
            return
        rng = rng if rng is not None else np.random.default_rng()
        new = (np.ascontiguousarray(levels, dtype=np.uint32) if levels is not None
               else hnsw_rand_levels(n - n_old, self.config.M, rng))
        if new.shape != (n - n_old,):
            raise ValueError("one level per new row is required")
        L.check(L.lib().vdb_hnsw_append(self._h, self.vec_set._h, L.ptr(new), self.MAX_BATCH))
        self.levels = np.concatenate([self.levels, new])

    def __len__(self):
        return len(self.vec_set)

    @property
    def enter_point(self):
        ep, el = C.c_int64(-1), C.c_int32(-1)
        L.check(L.lib().vdb_hnsw_info(self._h, None, None, None, C.byref(ep), C.byref(el)))
        return int(ep.value), int(el.value)

    def level0_links(self):
        """(links [n, 2M] u32, lengths [n] u32) as the reference stores them (hnsw_index.rs:110-112)."""
        n = len(self.vec_set)
        links = np.zeros((n, 2 * self.config.M), np.uint32)
        lens = np.zeros(n, np.uint32)
        L.check(L.lib().vdb_hnsw_links0(self._h, L.ptr(links), L.ptr(lens)))
        return links, lens

    def upper_links(self):
        """(levels [n], links [sum(levels) * M], lengths [sum(levels)]): other_links / links_len of the reference."""
        n = len(self.vec_set)
        levels = np.zeros(n, np.uint32)
        slots = int(self.levels.sum())
        ulinks = np.zeros(max(slots, 1) * self.config.M, np.uint32)
        ulen = np.zeros(max(slots, 1), np.uint32)
        L.check(L.lib().vdb_hnsw_upper(self._h, L.ptr(levels), L.ptr(ulinks), L.ptr(ulen)))
        return levels, ulinks[:slots * self.config.M], ulen[:slots]

    @classmethod
    def from_record(cls, vec_set: DeviceVecSet, rec):
        """IndexSerdeExternalVecSet::load_with_external_vec_set (hnsw_index.rs:656-668): the graph of a bincode
        HNSWIndex file (formats.load_hnsw_index) over the rows of `vec_set`."""
        n = len(vec_set)
        if len(rec.vec_level) != n or rec.dim != vec_set.dim:
            raise ValueError("the index file does not describe this vector set")
        self = cls.__new__(cls)
        self.vec_set = vec_set
        self.config = HNSWConfig(rec.max_elements, rec.ef_construction, rec.m)
        self.levels = np.asarray(rec.vec_level, np.uint32)
        links0 = np.ascontiguousarray(rec.level0_links, np.uint32).reshape(n, rec.max_m0)
        len0 = np.array([int(l[0]) for l in rec.links_len], np.uint32) if n else np.zeros(0, np.uint32)
        ulinks = (np.concatenate([np.asarray(o, np.uint32) for o in rec.other_links]) if n else np.zeros(0, np.uint32))
        ulen = (np.concatenate([np.asarray(l[1:], np.uint32) for l in rec.links_len]) if n else np.zeros(0, np.uint32))
        ulinks = np.ascontiguousarray(ulinks if ulinks.size else np.zeros(1, np.uint32), np.uint32)
        ulen = np.ascontiguousarray(ulen if ulen.size else np.zeros(1, np.uint32), np.uint32)
        self._h = C.c_void_p()
        L.check(L.lib().vdb_hnsw_create_from_graph(vec_set._h, rec.m, rec.ef_construction, L.ptr(self.levels), L.ptr(links0),
                                                   L.ptr(len0), L.ptr(ulinks), L.ptr(ulen),
                                                   -1 if rec.enter_point is None else rec.enter_point,
                                                   -1 if rec.enter_level is None else rec.enter_level, C.byref(self._h)))
        self.ef_construction = rec.ef_construction
        self.default_ef = rec.default_ef
        return self

    def set_default_ef(self, ef):
        if ef <= 0:
            raise ValueError("The search radius should be positive.")
        self.default_ef = ef

    def knn_with_ef_batch(self, queries, k, ef):
        vs = self.vec_set
        q = _as_rows(queries, vs.dtype)
        if q.shape[1] != vs.dim:
            raise ValueError("The dimension of the query doesn't match.")
        if ef <= 0:
            raise ValueError("The search radius should be positive.")
        nq = q.shape[0]
        ids = np.full((nq, k), np.iinfo(np.uint64).max, np.uint64)
        dist = np.full((nq, k), np.nan, np.float32)
        counts = np.zeros(nq, np.uint32)
        L.check(L.lib().vdb_hnsw_knn(vs._h, self._h, L.ptr(q), nq, k, ef, L.ptr(ids), L.ptr(dist), L.ptr(counts)))
        return ids, dist, counts

    def knn_with_ef(self, query, k, ef):
        """IndexKNNWithEf::knn_with_ef (hnsw_index.rs:616-625)."""
        return _pairs(*self.knn_with_ef_batch(np.asarray(query).reshape(1, -1), k, ef))[0]

    def knn(self, query, k):
        return self.knn_with_ef(query, k, self.default_ef)

    def knn_pq_batch(self, queries, k, ef, pq_table):
        vs = self.vec_set
        q = _as_rows(queries, vs.dtype)
        if q.shape[1] != vs.dim:
            raise ValueError("The dimension of the query doesn't match.")
        if ef <= 0:
            raise ValueError("The search radius should be positive.")
        nq = q.shape[0]
        ids = np.full((nq, k), np.iinfo(np.uint64).max, np.uint64)
        dist = np.full((nq, k), np.nan, np.float32)
        counts = np.zeros(nq, np.uint32)
        L.check(L.lib().vdb_hnsw_knn_pq(vs._h, self._h, pq_table._h, L.ptr(q), nq, k, ef, L.ptr(ids), L.ptr(dist),
                                        L.ptr(counts)))
        return ids, dist, counts

    def knn_pq(self, query, k, ef, pq_table):
        """IndexPQ::knn_pq (hnsw_index.rs:672-697)."""
        return _pairs(*self.knn_pq_batch(np.asarray(query).reshape(1, -1), k, ef, pq_table))[0]

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            L.lib().vdb_hnsw_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
