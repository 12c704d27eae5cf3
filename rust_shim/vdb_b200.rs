//! Source-only Rust binding of include/vdb_b200.h for lab-1806-vec-db v0.8.1. It cannot be compiled in the build
//! image (no Rust toolchain), so it is kept self-consistent by hand: every `extern "C"` item below is declared in
//! include/vdb_b200.h with the same argument order and widths (tests/test_host_cpu.py checks the names against the
//! built library), and it only touches items of the reference crate that exist at the cited lines.
//!
//! A maintainer adds this file as `src/gpu.rs` (it uses `pub(crate)` fields of `HNSWIndex`, so it lives inside the
//! crate), links `libvdb_b200.so` from build.rs (`println!("cargo:rustc-link-lib=dylib=vdb_b200")`) and swaps
//!   FlatIndex<T>  -> GpuFlatIndex<T>      (IndexKNN, IndexPQ, IndexFromVecSet;   src/index_algorithm/flat_index.rs)
//!   IVFIndex<T>   -> GpuIvfIndex<T>       (IndexKNN, IndexKNNWithEf, IndexPQ, IndexFromVecSet; ivf_index.rs)
//!   HNSWIndex<T>  -> GpuHnswIndex<T>      (IndexKNN, IndexKNNWithEf, IndexPQ, build_on_vec_set; hnsw_index.rs)
//!   KMeans::from_vec_set / find_nearest   -> gpu_kmeans_from_vec_set / gpu_find_nearest_batch (src/distance/k_means.rs)
//!   PQTable::from_vec_set                 -> gpu_pq_table_from_vec_set            (src/distance/pq_table.rs:141-191)
//! behind the same traits (src/index_algorithm/mod.rs:35-154). With `gpu_init(&[0,1,..,7])` called once, the same
//! `knn` call runs row-sharded on every listed GPU (one C call, per-GPU top-k merged over NVLink peer memory); HNSW
//! keeps a replica per GPU and splits the query batch over them.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};
use std::sync::Mutex;

use rand::{distributions::WeightedIndex, prelude::Distribution, Rng};

use crate::{
    distance::{
        k_means::{KMeans, KMeansConfig},
        pq_table::{pq_groups, PQConfig, PQTable},
        DistanceAlgorithm,
    },
    index_algorithm::{
        hnsw_index::{HNSWConfig, HNSWIndex},
        ivf_index::{IVFConfig, IVFIndex},
        prelude::*,
        CandidatePair,
    },
    scalar::Scalar,
    vec_set::VecSet,
};

#[repr(C)] pub struct vdb_dataset { _p: [u8; 0] }
#[repr(C)] pub struct vdb_pq { _p: [u8; 0] }
#[repr(C)] pub struct vdb_ivf { _p: [u8; 0] }
#[repr(C)] pub struct vdb_hnsw { _p: [u8; 0] }

extern "C" {
    pub fn vdb_last_error() -> *const c_char;
    pub fn vdb_init(devices: *const c_int, n: u32) -> c_int;
    pub fn vdb_dataset_create(rows: *const c_void, n: u64, dim: u32, dtype: c_int, metric: c_int,
                              id_base: u64, out: *mut *mut vdb_dataset) -> c_int;
    pub fn vdb_dataset_append(ds: *mut vdb_dataset, rows: *const c_void, n: u64) -> c_int;
    pub fn vdb_dataset_swap_remove(ds: *mut vdb_dataset, idx: u64) -> c_int;
    pub fn vdb_dataset_destroy(ds: *mut vdb_dataset) -> c_int;
    pub fn vdb_flat_knn(ds: *const vdb_dataset, queries: *const c_void, nq: u32, k: u32,
                        ids: *mut u64, dist: *mut f32, counts: *mut u32) -> c_int;
    pub fn vdb_pq_create(ds: *const vdb_dataset, codebooks: *const c_void, m: u32, n_bits: u32,
                         codes: *mut u8, out: *mut *mut vdb_pq) -> c_int;
    pub fn vdb_pq_create_from_codes(ds: *const vdb_dataset, codebooks: *const c_void, m: u32, n_bits: u32,
                                    codes: *const u8, out: *mut *mut vdb_pq) -> c_int;
    pub fn vdb_pq_destroy(pq: *mut vdb_pq) -> c_int;
    pub fn vdb_pq_knn(ds: *const vdb_dataset, pq: *const vdb_pq, queries: *const c_void, nq: u32, k: u32,
                      ef: u32, ids: *mut u64, dist: *mut f32, counts: *mut u32) -> c_int;
    pub fn vdb_pq_train_ds(train: *const vdb_dataset, m: u32, n_bits: u32, max_iter: u32, tol: f32,
                           uniforms: *const f64, init_codebooks: *const c_void, codebooks: *mut c_void,
                           iters: *mut u32) -> c_int;
    pub fn vdb_kmeans_assign(rows: *const c_void, n: u64, dim: u32, dtype: c_int, metric: c_int,
                             centroids: *const c_void, k: u32, sel_lo: u32, sel_hi: u32, out: *mut u32) -> c_int;
    pub fn vdb_kmeans_train(rows: *const c_void, n: u64, dim: u32, dtype: c_int, metric: c_int,
                            centroids: *mut c_void, k: u32, sel_lo: u32, sel_hi: u32, max_iter: u32,
                            tol: f32, iters: *mut u32) -> c_int;
    pub fn vdb_kmeans_pp_weights(rows: *const c_void, n: u64, dim: u32, dtype: c_int, metric: c_int,
                                 centroid: *const c_void, sel_lo: u32, sel_hi: u32, weights: *mut f32) -> c_int;
    pub fn vdb_ivf_create(ds: *const vdb_dataset, centroids: *const c_void, nlist: u32,
                          assign_out: *mut u32, out: *mut *mut vdb_ivf) -> c_int;
    pub fn vdb_ivf_destroy(ivf: *mut vdb_ivf) -> c_int;
    pub fn vdb_ivf_knn(ds: *const vdb_dataset, ivf: *const vdb_ivf, queries: *const c_void, nq: u32, k: u32,
                       n_probes: u32, ids: *mut u64, dist: *mut f32, counts: *mut u32) -> c_int;
    pub fn vdb_ivf_knn_pq(ds: *const vdb_dataset, ivf: *const vdb_ivf, pq: *const vdb_pq, queries: *const c_void, nq: u32,
                          k: u32, ef: u32, n_probes: u32, ids: *mut u64, dist: *mut f32, counts: *mut u32) -> c_int;
    pub fn vdb_hnsw_build(ds: *const vdb_dataset, m: u32, ef_construction: u32, levels: *const u32, max_batch: u32,
                          out: *mut *mut vdb_hnsw) -> c_int;
    pub fn vdb_hnsw_destroy(h: *mut vdb_hnsw) -> c_int;
    pub fn vdb_hnsw_append(h: *mut vdb_hnsw, ds: *const vdb_dataset, new_levels: *const u32, max_batch: u32) -> c_int;
    pub fn vdb_hnsw_info(h: *const vdb_hnsw, n: *mut u64, m: *mut u32, ef_construction: *mut u32,
                         enter_point: *mut i64, enter_level: *mut i32) -> c_int;
    pub fn vdb_hnsw_knn(ds: *const vdb_dataset, h: *const vdb_hnsw, queries: *const c_void, nq: u32, k: u32, ef: u32,
                        ids: *mut u64, dist: *mut f32, counts: *mut u32) -> c_int;
    pub fn vdb_hnsw_knn_pq(ds: *const vdb_dataset, h: *const vdb_hnsw, pq: *const vdb_pq, queries: *const c_void, nq: u32,
                           k: u32, ef: u32, ids: *mut u64, dist: *mut f32, counts: *mut u32) -> c_int;
    pub fn vdb_hnsw_links0(h: *const vdb_hnsw, links0: *mut u32, len0: *mut u32) -> c_int;
    pub fn vdb_hnsw_upper(h: *const vdb_hnsw, levels: *mut u32, ulinks: *mut u32, ulen: *mut u32) -> c_int;
    pub fn vdb_hnsw_create_from_graph(ds: *const vdb_dataset, m: u32, ef_construction: u32, levels: *const u32,
                                      links0: *const u32, len0: *const u32, ulinks: *const u32, ulen: *const u32,
                                      enter_point: i64, enter_level: i32, out: *mut *mut vdb_hnsw) -> c_int;
    pub fn vdb_gather_dist(ds: *const vdb_dataset, queries: *const c_void, nq: u32, cand_ids: *const u32,
                           cand_off: *const u64, out: *mut f32) -> c_int;
    pub fn vdb_row_cache(ds: *const vdb_dataset, out: *mut f32) -> c_int;
    pub fn vdb_calc_dist(a: *const c_void, b: *const c_void, count: u64, dim: u32, dtype: c_int,
                         metric: c_int, out: *mut f32) -> c_int;
}

fn check(rc: c_int) {
    // the reference's trait methods are infallible and panic on misuse (assert!), so does the shim
    if rc != 0 {
        let msg = unsafe { std::ffi::CStr::from_ptr(vdb_last_error()) }.to_string_lossy().into_owned();
        panic!("vdb_b200 error {rc}: {msg}");
    }
}
fn dtype_of<T: Scalar>() -> c_int { if std::mem::size_of::<T>() == 4 { 0 } else { 1 } } // Scalar = f32 | u8 (scalar.rs:117-119)
fn metric_of(d: DistanceAlgorithm) -> c_int { match d { DistanceAlgorithm::L2Sqr => 0, DistanceAlgorithm::Cosine => 1 } }
/// `VecSet::data` is private (vec_set.rs:15-20); rows are contiguous, so row 0's pointer is the whole block's.
fn rows_ptr<T: Scalar>(vs: &VecSet<T>) -> *const c_void {
    if vs.is_empty() { std::ptr::null() } else { vs[0].as_ptr() as *const c_void }
}
fn flat_rows<T: Scalar>(vs: &VecSet<T>) -> Vec<T> { vs.iter().flat_map(|v| v.iter().copied()).collect() }

/// Registers the GPUs of this process (SURVEY.md 8b `vdb_init`): with two or more, datasets created afterwards are
/// row-sharded over them and every search stays ONE call (index_algorithm/mod.rs:84-91).
pub fn gpu_init(devices: &[i32]) { check(unsafe { vdb_init(devices.as_ptr(), devices.len() as u32) }); }

fn pairs(ids: &[u64], dist: &[f32], count: u32) -> Vec<CandidatePair> {
    (0..count as usize).map(|j| CandidatePair::new(ids[j] as usize, dist[j])).collect()
}

/// Owned device mirror of one `VecSet<T>`; host memory stays authoritative.
struct Mirror(*mut vdb_dataset);
unsafe impl Send for Mirror {}
unsafe impl Sync for Mirror {} // vdb_*_knn are re-entrant on one handle (include/vdb_b200.h, conventions)
impl Mirror {
    fn of<T: Scalar>(vs: &VecSet<T>, dist: DistanceAlgorithm) -> Self {
        let mut ds = std::ptr::null_mut();
        check(unsafe { vdb_dataset_create(rows_ptr(vs), vs.len() as u64, vs.dim() as u32, dtype_of::<T>(),
                                          metric_of(dist), 0, &mut ds) });
        Mirror(ds)
    }
}
impl Drop for Mirror { fn drop(&mut self) { unsafe { vdb_dataset_destroy(self.0); } } }

/// Device mirror of a `PQTable<T>` over the rows of one dataset, keyed by the address of the table's code block:
/// the reference drops the PQ table on every write (metadata_vec_table.rs:65, 77, 171), so a new table is a new key.
struct PqMirror { key: (usize, usize), pq: *mut vdb_pq }
unsafe impl Send for PqMirror {}
impl Drop for PqMirror { fn drop(&mut self) { unsafe { vdb_pq_destroy(self.pq); } } }

fn pq_mirror<T: Scalar>(slot: &Mutex<Option<PqMirror>>, ds: *mut vdb_dataset, t: &PQTable<T>) -> *mut vdb_pq {
    let key = (rows_ptr(&t.encoded_vec_set) as usize, t.encoded_vec_set.len());
    let mut g = slot.lock().unwrap();
    if g.as_ref().map(|m| m.key) != Some(key) {
        // codebooks: group g = [k, len_g] rows of T, groups concatenated (PQTable::group_k_means, pq_table.rs:131-132)
        let books: Vec<T> = t.group_k_means.iter().flat_map(|km| flat_rows(&km.centroids)).collect();
        let mut pq = std::ptr::null_mut();
        check(unsafe { vdb_pq_create_from_codes(ds, books.as_ptr() as _, t.config.m as u32, t.config.n_bits as u32,
                                                rows_ptr(&t.encoded_vec_set) as *const u8, &mut pq) });
        *g = Some(PqMirror { key, pq });
    }
    g.as_ref().unwrap().pq
}

// ------------------------------------------------------------------------------------------------ Flat
/// Drop-in for `FlatIndex<T>` (flat_index.rs:21-27).
pub struct GpuFlatIndex<T: Scalar> {
    pub dist: DistanceAlgorithm,
    pub vec_set: VecSet<T>,
    ds: Mirror,
    pq: Mutex<Option<PqMirror>>,
}
impl<T: Scalar> GpuFlatIndex<T> {
    /// Additive batch entry (the trait call is nq == 1); `queries` is nq x dim, row-major.
    pub fn knn_batch(&self, queries: &[T], nq: usize, k: usize) -> Vec<Vec<CandidatePair>> {
        let (mut ids, mut dist, mut cnt) = (vec![0u64; nq * k], vec![0f32; nq * k], vec![0u32; nq]);
        check(unsafe { vdb_flat_knn(self.ds.0, queries.as_ptr() as _, nq as u32, k as u32,
                                    ids.as_mut_ptr(), dist.as_mut_ptr(), cnt.as_mut_ptr()) });
        (0..nq).map(|q| pairs(&ids[q * k..(q + 1) * k], &dist[q * k..(q + 1) * k], cnt[q])).collect()
    }
    /// VecSet::push / swap_remove keep the mirror in step (dynamic_index.rs:49-56, metadata_vec_table.rs:180-185).
    pub fn push(&mut self, v: &[T]) -> usize {
        check(unsafe { vdb_dataset_append(self.ds.0, v.as_ptr() as _, 1) });
        self.vec_set.push(v)
    }
    pub fn swap_remove(&mut self, idx: usize) {
        check(unsafe { vdb_dataset_swap_remove(self.ds.0, idx as u64) });
        self.vec_set.swap_remove(idx);
    }
}
impl<T: Scalar> std::ops::Index<usize> for GpuFlatIndex<T> {
    type Output = [T];
    fn index(&self, i: usize) -> &[T] { &self.vec_set[i] }
}
impl<T: Scalar> IndexIter<T> for GpuFlatIndex<T> {
    fn dim(&self) -> usize { self.vec_set.dim() }
    fn len(&self) -> usize { self.vec_set.len() }
}
impl<T: Scalar> IndexFromVecSet<T> for GpuFlatIndex<T> {
    type Config = ();
    fn from_vec_set(vec_set: VecSet<T>, dist: DistanceAlgorithm, _: (), _: &mut impl Rng) -> Self {
        let ds = Mirror::of(&vec_set, dist);
        Self { dist, vec_set, ds, pq: Mutex::new(None) }
    }
}
impl<T: Scalar> IndexKNN<T> for GpuFlatIndex<T> {
    /// replaces FlatIndex::knn (flat_index.rs:48-57). Concurrent calls from rayon workers (examples/bench.rs:410-416)
    /// are coalesced into shared database passes inside the library.
    fn knn(&self, query: &[T], k: usize) -> Vec<CandidatePair> { self.knn_batch(query, 1, k).pop().unwrap() }
}
impl<T: Scalar> IndexPQ<T> for GpuFlatIndex<T> {
    /// replaces FlatIndex::knn_pq (flat_index.rs:84-104)
    fn knn_pq(&self, query: &[T], k: usize, ef: usize, pq_table: &PQTable<T>) -> Vec<CandidatePair> {
        assert_eq!(self.dist, pq_table.config.dist, "Distance algorithm mismatch."); // flat_index.rs:92-95
        let pq = pq_mirror(&self.pq, self.ds.0, pq_table);
        let (mut ids, mut dist, mut cnt) = (vec![0u64; k], vec![0f32; k], vec![0u32; 1]);
        check(unsafe { vdb_pq_knn(self.ds.0, pq, query.as_ptr() as _, 1, k as u32, ef as u32,
                                  ids.as_mut_ptr(), dist.as_mut_ptr(), cnt.as_mut_ptr()) });
        pairs(&ids, &dist, cnt[0])
    }
}

// ------------------------------------------------------------------------------------------------ k-means
/// KMeans::from_vec_set (k_means.rs:95-162): k-means++ draws stay on the host with the CALLER's rng, in the
/// reference's order (first = gen_range(0..n); then WeightedIndex over the weights, with the uniform fallback drawn
/// eagerly every round, k_means.rs:71-82); the weight update (:75-77), the assignment (:117-120) and the Lloyd update
/// (:121-161) run on the GPU with the reference's arithmetic (bit-exact given the initial centroids).
pub fn gpu_kmeans_from_vec_set<T: Scalar>(vec_set: &VecSet<T>, config: KMeansConfig, rng: &mut impl Rng) -> KMeans<T> {
    assert!(config.k > 0, "The number of clusters should be greater than 0.");
    assert!(config.selected.is_none() || config.selected.as_ref().unwrap().end <= vec_set.dim(),
            "The selected range should be in the range [0, vec_set.dim())");
    let (l, r) = match &config.selected { Some(s) => (s.start, s.end), None => (0, vec_set.dim()) };
    let (n, dim, sub) = (vec_set.len(), vec_set.dim(), r - l);
    let (dt, me) = (dtype_of::<T>(), metric_of(config.dist));
    let mut cent: Vec<T> = Vec::with_capacity(config.k * sub);
    let first = rng.gen_range(0..n);
    cent.extend_from_slice(&vec_set[first][l..r]);
    let mut weight = vec![f32::INFINITY; n];
    for idx in 1..config.k {
        check(unsafe { vdb_kmeans_pp_weights(rows_ptr(vec_set), n as u64, dim as u32, dt, me,
                                             cent[(idx - 1) * sub..].as_ptr() as _, l as u32, r as u32,
                                             weight.as_mut_ptr()) });
        let c = WeightedIndex::new(&weight).map(|d| d.sample(rng)).unwrap_or(rng.gen_range(0..n));
        cent.extend_from_slice(&vec_set[c][l..r]);
    }
    let mut iters = 0u32;
    check(unsafe { vdb_kmeans_train(rows_ptr(vec_set), n as u64, dim as u32, dt, me, cent.as_mut_ptr() as _,
                                    config.k as u32, l as u32, r as u32, config.max_iter as u32, config.tol, &mut iters) });
    KMeans { config, centroids: VecSet::new(sub, cent) }
}
/// KMeans::find_nearest (k_means.rs:166-170) for every row of `rows` at once (the rayon map of ivf_index.rs:89-93).
pub fn gpu_find_nearest_batch<T: Scalar>(km: &KMeans<T>, rows: &VecSet<T>) -> Vec<usize> {
    let (l, r) = match &km.config.selected { Some(s) => (s.start, s.end), None => (0, rows.dim()) };
    let mut out = vec![0u32; rows.len()];
    check(unsafe { vdb_kmeans_assign(rows_ptr(rows), rows.len() as u64, rows.dim() as u32, dtype_of::<T>(),
                                     metric_of(km.config.dist), rows_ptr(&km.centroids), km.config.k as u32,
                                     l as u32, r as u32, out.as_mut_ptr()) });
    out.into_iter().map(|c| c as usize).collect()
}

// ------------------------------------------------------------------------------------------------ PQ table
/// PQTable::from_vec_set (pq_table.rs:141-191): sample (:146-148), one k-means per group (:154-172; the host loop keeps
/// the rng stream of the reference), dist_cache (:165-170), and the encode loop (:178-181) as one GPU pass.
pub fn gpu_pq_table_from_vec_set<T: Scalar>(vec_set: &VecSet<T>, config: PQConfig, rng: &mut impl Rng) -> PQTable<T> {
    assert!(config.n_bits == 4 || config.n_bits == 8, "n_bits must be 4 or 8 in PQTable.");
    let (m, k, dim) = (config.m, 1usize << config.n_bits, vec_set.dim());
    let sub_vec_set = config.k_means_size.map(|size| vec_set.random_sample(size, rng));
    let train = sub_vec_set.as_ref().unwrap_or(vec_set);
    let mut group_k_means = Vec::with_capacity(m);
    let mut dist_cache = Vec::with_capacity(m * k);
    for selected in pq_groups(dim, m) {
        let cfg = KMeansConfig { k, max_iter: config.k_means_max_iter, tol: config.k_means_tol, dist: config.dist,
                                 selected: Some(selected) };
        let km = gpu_kmeans_from_vec_set(train, cfg, rng);
        for c in km.centroids.iter() {
            dist_cache.push(match config.dist { DistanceAlgorithm::L2Sqr => 0.0, DistanceAlgorithm::Cosine => T::dot_product(c, c) });
        }
        group_k_means.push(km);
    }
    let encoded_dim = if config.n_bits == 4 { m.div_ceil(2) } else { m };
    let books: Vec<T> = group_k_means.iter().flat_map(|km| flat_rows(&km.centroids)).collect();
    let mut codes = vec![0u8; vec_set.len() * encoded_dim];
    let ds = Mirror::of(vec_set, config.dist);
    let mut pq = std::ptr::null_mut();
    check(unsafe { vdb_pq_create(ds.0, books.as_ptr() as _, m as u32, config.n_bits as u32, codes.as_mut_ptr(), &mut pq) });
    unsafe { vdb_pq_destroy(pq); } // the search-side mirror is rebuilt from the codes by the index that uses the table
    PQTable { config, dim, k, encoded_dim, encoded_vec_set: VecSet::new(encoded_dim, codes), group_k_means, dist_cache }
}

// ------------------------------------------------------------------------------------------------ IVF
/// Drop-in for `IVFIndex<T>` (ivf_index.rs:34-47): the host struct is kept whole (serde, `clusters`), the probe scan
/// runs on the device mirror.
pub struct GpuIvfIndex<T: Scalar> {
    pub inner: IVFIndex<T>,
    ds: Mirror,
    ivf: *mut vdb_ivf,
    pq: Mutex<Option<PqMirror>>,
}
unsafe impl<T: Scalar> Send for GpuIvfIndex<T> {}
unsafe impl<T: Scalar> Sync for GpuIvfIndex<T> {}
impl<T: Scalar> Drop for GpuIvfIndex<T> { fn drop(&mut self) { unsafe { vdb_ivf_destroy(self.ivf); } } }
impl<T: Scalar> std::ops::Index<usize> for GpuIvfIndex<T> {
    type Output = [T];
    fn index(&self, i: usize) -> &[T] { &self.inner.vec_set[i] }
}
impl<T: Scalar> IndexIter<T> for GpuIvfIndex<T> {
    fn dim(&self) -> usize { self.inner.vec_set.dim() }
    fn len(&self) -> usize { self.inner.vec_set.len() }
}
impl<T: Scalar> IndexFromVecSet<T> for GpuIvfIndex<T> {
    type Config = IVFConfig;
    /// replaces IVFIndex::from_vec_set (ivf_index.rs:67-107)
    fn from_vec_set(vec_set: VecSet<T>, dist: DistanceAlgorithm, config: IVFConfig, rng: &mut impl Rng) -> Self {
        let k = config.k;
        let kc = KMeansConfig { k, max_iter: config.k_means_max_iter, tol: config.k_means_tol, dist, selected: None };
        let k_means = match config.k_means_size {
            Some(size) => gpu_kmeans_from_vec_set(&vec_set.random_sample(size, rng), kc, rng),
            None => gpu_kmeans_from_vec_set(&vec_set, kc, rng),
        };
        let ds = Mirror::of(&vec_set, dist);
        let mut assign = vec![0u32; vec_set.len()];
        let mut ivf = std::ptr::null_mut();
        check(unsafe { vdb_ivf_create(ds.0, rows_ptr(&k_means.centroids), k as u32, assign.as_mut_ptr(), &mut ivf) });
        let mut clusters = vec![vec![]; k];
        for (i, &c) in assign.iter().enumerate() { clusters[c as usize].push(i); }
        Self { inner: IVFIndex { dist, default_n_probes: 4, vec_set, config, clusters, k_means }, ds, ivf, pq: Mutex::new(None) }
    }
}
impl<T: Scalar> IndexKNN<T> for GpuIvfIndex<T> {
    fn knn(&self, query: &[T], k: usize) -> Vec<CandidatePair> { self.knn_with_ef(query, k, self.inner.default_n_probes) }
}
impl<T: Scalar> IndexKNNWithEf<T> for GpuIvfIndex<T> {
    fn set_default_ef(&mut self, n_probes: usize) { self.inner.default_n_probes = n_probes; }
    /// replaces IVFIndex::knn_with_ef (ivf_index.rs:143-154); `ef` is the number of probes
    fn knn_with_ef(&self, query: &[T], k: usize, n_probes: usize) -> Vec<CandidatePair> {
        let (mut ids, mut dist, mut cnt) = (vec![0u64; k], vec![0f32; k], vec![0u32; 1]);
        check(unsafe { vdb_ivf_knn(self.ds.0, self.ivf, query.as_ptr() as _, 1, k as u32, n_probes as u32,
                                   ids.as_mut_ptr(), dist.as_mut_ptr(), cnt.as_mut_ptr()) });
        pairs(&ids, &dist, cnt[0])
    }
}

impl<T: Scalar> IndexPQ<T> for GpuIvfIndex<T> {
    /// IVF knn_pq (the reference has none; INTEGRATION.md defines it): FlatIndex::knn_pq (flat_index.rs:84-104)
    /// restricted to the rows of the default_n_probes nearest lists
    fn knn_pq(&self, query: &[T], k: usize, ef: usize, pq_table: &PQTable<T>) -> Vec<CandidatePair> {
        assert_eq!(self.inner.dist, pq_table.config.dist, "Distance algorithm mismatch.");
        let pq = pq_mirror(&self.pq, self.ds.0, pq_table);
        let (mut ids, mut dist, mut cnt) = (vec![0u64; k], vec![0f32; k], vec![0u32; 1]);
        check(unsafe { vdb_ivf_knn_pq(self.ds.0, self.ivf, pq, query.as_ptr() as _, 1, k as u32, ef as u32,
                                      self.inner.default_n_probes as u32, ids.as_mut_ptr(), dist.as_mut_ptr(),
                                      cnt.as_mut_ptr()) });
        pairs(&ids, &dist, cnt[0])
    }
}

// ------------------------------------------------------------------------------------------------ HNSW
/// Drop-in for `HNSWIndex<T>` (hnsw_index.rs:99-141). The graph lives on the device in the reference's own layout;
/// `to_host` copies it into an `HNSWIndex<T>` (bincode save, IndexSerdeExternalVecSet :641-668) and `from_host`
/// mirrors a loaded one. After `gpu_init` with several GPUs every GPU holds a replica of the rows and the graph, and each
/// `knn` / `knn_pq` batch is split over them in one call, with the single-GPU results; `batch_add` is refused there.
pub struct GpuHnswIndex<T: Scalar> {
    pub dist: DistanceAlgorithm,
    pub vec_set: VecSet<T>,
    pub config: HNSWConfig,
    pub default_ef: usize,
    ds: Mirror,
    h: *mut vdb_hnsw,
    pq: Mutex<Option<PqMirror>>,
}
unsafe impl<T: Scalar> Send for GpuHnswIndex<T> {}
unsafe impl<T: Scalar> Sync for GpuHnswIndex<T> {}
impl<T: Scalar> Drop for GpuHnswIndex<T> { fn drop(&mut self) { unsafe { vdb_hnsw_destroy(self.h); } } }

/// rand_level (hnsw_index.rs:145-149) with the caller's rng, one draw per row in row order.
fn rand_levels(n: usize, m: usize, rng: &mut impl Rng) -> Vec<u32> {
    let inv_log_m = 1.0 / (m as f32).ln();
    (0..n).map(|_| { let u: f32 = rng.gen_range(0.0..1.0); (-u.ln() * inv_log_m).floor() as u32 }).collect()
}
const MAX_BATCH: u32 = 2048; // upper bound of next_batch_size (hnsw_index.rs:389-395) on the device

impl<T: Scalar> GpuHnswIndex<T> {
    /// IndexBuilder::build_on_vec_set (hnsw_index.rs:585-600)
    pub fn build_on_vec_set(vec_set: VecSet<T>, dist: DistanceAlgorithm, config: HNSWConfig, rng: &mut impl Rng) -> Self {
        let ds = Mirror::of(&vec_set, dist);
        let levels = rand_levels(vec_set.len(), config.M, rng);
        let mut h = std::ptr::null_mut();
        check(unsafe { vdb_hnsw_build(ds.0, config.M as u32, config.ef_construction as u32, levels.as_ptr(), MAX_BATCH, &mut h) });
        let default_ef = config.ef_construction.max(2 * config.M) / 2; // hnsw_index.rs:495-506
        Self { dist, vec_set, config, default_ef, ds, h, pq: Mutex::new(None) }
    }
    /// IndexBuilder::batch_add (hnsw_index.rs:563-575)
    pub fn batch_add(&mut self, vec_list: &[&[T]], rng: &mut impl Rng) -> Vec<usize> {
        let first = self.vec_set.len();
        for v in vec_list {
            check(unsafe { vdb_dataset_append(self.ds.0, v.as_ptr() as _, 1) });
            self.vec_set.push(v);
        }
        let levels = rand_levels(vec_list.len(), self.config.M, rng);
        check(unsafe { vdb_hnsw_append(self.h, self.ds.0, levels.as_ptr(), MAX_BATCH) });
        (first..first + vec_list.len()).collect()
    }
    /// Mirrors an index loaded from the reference's bincode file (HNSWIndex::load_with_external_vec_set :656-668).
    pub fn from_host(idx: HNSWIndex<T>) -> Self {
        let n = idx.vec_set.len();
        let (m, m0) = (idx.config.m, idx.config.max_m0);
        let levels: Vec<u32> = idx.vec_level.iter().map(|&l| l as u32).collect();
        let len0: Vec<u32> = (0..n).map(|i| idx.links_len[i][0] as u32).collect();
        let (mut ulinks, mut ulen) = (Vec::new(), Vec::new());
        for i in 0..n {
            ulinks.extend_from_slice(&idx.other_links[i][..idx.vec_level[i] * m]);
            ulen.extend(idx.links_len[i][1..].iter().map(|&l| l as u32));
        }
        debug_assert_eq!(idx.level0_links.len(), n * m0);
        let ds = Mirror::of(&idx.vec_set, idx.config.dist);
        let mut h = std::ptr::null_mut();
        check(unsafe { vdb_hnsw_create_from_graph(ds.0, m as u32, idx.config.ef_construction as u32, levels.as_ptr(),
                                                  idx.level0_links.as_ptr(), len0.as_ptr(), ulinks.as_ptr(), ulen.as_ptr(),
                                                  idx.enter_point.map_or(-1, |p| p as i64),
                                                  idx.enter_level.map_or(0, |l| l as i32), &mut h) });
        let config = HNSWConfig { max_elements: idx.config.max_elements, ef_construction: idx.config.ef_construction, M: m };
        Self { dist: idx.config.dist, default_ef: idx.config.default_ef, vec_set: idx.vec_set, config, ds, h, pq: Mutex::new(None) }
    }
    /// Copies the device graph into `host` (an `HNSWIndex::new` of the same dim / dist / config): level0_links,
    /// other_links, links_len, vec_level, enter point; `host.init_after_load()` then rebuilds dist_cache (:371-379).
    pub fn to_host(&self, host: &mut HNSWIndex<T>) {
        let (n, m) = (self.vec_set.len(), self.config.M);
        let (mut ep, mut el) = (0i64, 0i32);
        check(unsafe { vdb_hnsw_info(self.h, std::ptr::null_mut(), std::ptr::null_mut(), std::ptr::null_mut(), &mut ep, &mut el) });
        let (mut l0, mut len0) = (vec![0u32; n * 2 * m], vec![0u32; n]);
        check(unsafe { vdb_hnsw_links0(self.h, l0.as_mut_ptr(), len0.as_mut_ptr()) });
        let mut levels = vec![0u32; n];
        check(unsafe { vdb_hnsw_upper(self.h, levels.as_mut_ptr(), std::ptr::null_mut(), std::ptr::null_mut()) });
        let total: usize = levels.iter().map(|&l| l as usize).sum();
        let (mut ul, mut ulen) = (vec![0u32; total * m], vec![0u32; total]);
        check(unsafe { vdb_hnsw_upper(self.h, std::ptr::null_mut(), ul.as_mut_ptr(), ulen.as_mut_ptr()) });
        host.vec_set = self.vec_set.clone();
        host.level0_links = l0;
        host.vec_level = levels.iter().map(|&l| l as usize).collect();
        host.other_links.clear();
        host.links_len.clear();
        let mut at = 0usize;
        for i in 0..n {
            let lv = levels[i] as usize;
            host.other_links.push(ul[at * m..(at + lv) * m].to_vec());
            let mut ll = vec![len0[i] as usize];
            ll.extend(ulen[at..at + lv].iter().map(|&x| x as usize));
            host.links_len.push(ll);
            at += lv;
        }
        host.enter_point = if ep < 0 { None } else { Some(ep as usize) };
        host.enter_level = if ep < 0 { None } else { Some(el as usize) };
        host.init_after_load();
    }
}
impl<T: Scalar> std::ops::Index<usize> for GpuHnswIndex<T> {
    type Output = [T];
    fn index(&self, i: usize) -> &[T] { &self.vec_set[i] }
}
impl<T: Scalar> IndexIter<T> for GpuHnswIndex<T> {
    fn dim(&self) -> usize { self.vec_set.dim() }
    fn len(&self) -> usize { self.vec_set.len() }
}
impl<T: Scalar> IndexKNN<T> for GpuHnswIndex<T> {
    fn knn(&self, query: &[T], k: usize) -> Vec<CandidatePair> { self.knn_with_ef(query, k, self.default_ef) }
}
impl<T: Scalar> IndexKNNWithEf<T> for GpuHnswIndex<T> {
    fn set_default_ef(&mut self, ef: usize) {
        assert!(ef > 0, "The search radius should be positive.");
        self.default_ef = ef;
    }
    /// replaces HNSWIndex::knn_with_ef (hnsw_index.rs:616-625)
    fn knn_with_ef(&self, query: &[T], k: usize, ef: usize) -> Vec<CandidatePair> {
        if self.len() == 0 { return Vec::new(); }
        let (mut ids, mut dist, mut cnt) = (vec![0u64; k], vec![0f32; k], vec![0u32; 1]);
        check(unsafe { vdb_hnsw_knn(self.ds.0, self.h, query.as_ptr() as _, 1, k as u32, ef as u32,
                                    ids.as_mut_ptr(), dist.as_mut_ptr(), cnt.as_mut_ptr()) });
        pairs(&ids, &dist, cnt[0])
    }
}
impl<T: Scalar> IndexPQ<T> for GpuHnswIndex<T> {
    /// replaces HNSWIndex::knn_pq (hnsw_index.rs:672-697)
    fn knn_pq(&self, query: &[T], k: usize, ef: usize, pq_table: &PQTable<T>) -> Vec<CandidatePair> {
        if self.len() == 0 { return Vec::new(); }
        assert_eq!(self.dist, pq_table.config.dist, "Distance algorithm mismatch.");
        let pq = pq_mirror(&self.pq, self.ds.0, pq_table);
        let (mut ids, mut dist, mut cnt) = (vec![0u64; k], vec![0f32; k], vec![0u32; 1]);
        check(unsafe { vdb_hnsw_knn_pq(self.ds.0, self.h, pq, query.as_ptr() as _, 1, k as u32, ef as u32,
                                       ids.as_mut_ptr(), dist.as_mut_ptr(), cnt.as_mut_ptr()) });
        pairs(&ids, &dist, cnt[0])
    }
}

/// pyo3 `calc_dist` (src/pyo3/mod.rs:43-48) for `count` pairs at once.
pub fn gpu_calc_dist<T: Scalar>(a: &[T], b: &[T], dim: usize, dist: DistanceAlgorithm) -> Vec<f32> {
    assert_eq!(a.len(), b.len());
    let count = a.len() / dim;
    let mut out = vec![0f32; count];
    check(unsafe { vdb_calc_dist(a.as_ptr() as _, b.as_ptr() as _, count as u64, dim as u32, dtype_of::<T>(),
                                 metric_of(dist), out.as_mut_ptr()) });
    out
}
