/*
 * oracle.cpp — CPU restatement of lab-1806-vec-db v0.8.1's search hot path.
 *
 * TEST INFRASTRUCTURE ONLY (see oracle.h). Citations are relative to /root/reference/.
 * Arithmetic contract: rustc never contracts mul+add into FMA and never reassociates
 * float adds, so every reduction below is a plain left-to-right loop and this file MUST be
 * compiled with -ffp-contract=off and without -ffast-math (oracle/Makefile does that; the
 * `volatile`-free loops stay scalar because the compiler cannot reorder a float add chain).
 *
 * PARITY STATUS: pinned against the reference's RNG-free known-answer tests and against an
 * independent numpy float32 emulation on the reference's fixtures (tests/golden/). The Rust
 * crate itself cannot be built in this image. RNG-dependent steps (k-means++ draws,
 * random_sample) are "parity unpinned": rand 0.8.5 StdRng (ChaCha12) is not restated.
 */
#include "oracle.h"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstring>
#include <limits>
#include <set>
#include <thread>
#include <utility>
#include <vector>

namespace {

/* ---- scalar.rs:19-46: `as` casts ---------------------------------------------------- */
template <class T> inline float to_f32(T v) { return static_cast<float>(v); }
template <class T> inline T from_f32(float v);
template <> inline float from_f32<float>(float v) { return v; }
template <> inline uint8_t from_f32<uint8_t>(float v) {
    if (std::isnan(v)) return 0;            /* NaN -> 0 */
    if (v <= 0.0f) return 0;                /* saturate low (also truncation of (-1,0)) */
    if (v >= 255.0f) return 255;            /* saturate high */
    return static_cast<uint8_t>(v);         /* truncate toward zero */
}

/* ---- distance/mod.rs:72-95: sequential f32 reductions -------------------------------- */
template <class T> float dot(const T* a, const T* b, size_t n) {
    float s = 0.0f;
    for (size_t i = 0; i < n; ++i) {
        float p = to_f32(a[i]) * to_f32(b[i]);
        s = s + p;
    }
    return s;
}
template <class T> float l2sqr(const T* a, const T* b, size_t n) {
    float s = 0.0f;
    for (size_t i = 0; i < n; ++i) {
        float d = to_f32(a[i]) - to_f32(b[i]);
        float p = d * d;
        s = s + p;
    }
    return s;
}
/* distance/mod.rs:46-48 */
template <class T> float vec_norm(const T* a, size_t n) { return std::sqrt(dot(a, a, n)); }
/* f32::max semantics: NaN-ignoring */
inline float rmax(float a, float b) { return std::fmax(a, b); }
/* distance/mod.rs:54-57: ip_a + ip_b - 2.0 * dot, evaluated (ip_a + ip_b) - (2*dot) */
template <class T> float l2sqr_cached(const T* a, const T* b, size_t n, float ipa, float ipb) {
    float s = ipa + ipb;
    float t = 2.0f * dot(a, b, n);
    return s - t;
}
/* distance/mod.rs:67-69 */
template <class T> float cosine_cached(const T* a, const T* b, size_t n, float na, float nb) {
    float den = rmax(na * nb, 1e-10f);
    float q = dot(a, b, n) / den;
    return 1.0f - q;
}
/* distance/mod.rs:60-64 */
template <class T> float cosine(const T* a, const T* b, size_t n) {
    float na = vec_norm(a, n);
    float nb = vec_norm(b, n);
    return cosine_cached(a, b, n, na, nb);
}
/* distance/mod.rs:106-113 */
template <class T> float dist(const T* a, const T* b, size_t n, int metric) {
    return metric == ORC_L2SQR ? l2sqr(a, b, n) : cosine(a, b, n);
}

/* ---- candidate_pair.rs:10-40: CandidatePair ordered by (OrderedFloat distance, index) -- */
struct Pair {
    float d;
    uint64_t i;
};
/* ordered-float 4.2.2: total order, NaN == NaN and NaN greater than everything, -0 == +0 */
inline int cmp_of(float a, float b) {
    bool an = std::isnan(a), bn = std::isnan(b);
    if (an || bn) return an == bn ? 0 : (an ? 1 : -1);
    return a < b ? -1 : (a > b ? 1 : 0);
}
struct PairLess {
    bool operator()(const Pair& x, const Pair& y) const {
        int c = cmp_of(x.d, y.d);
        if (c != 0) return c < 0;
        return x.i < y.i;
    }
};
/* candidate_pair.rs:43-82: ResultSet (BTreeSet, bounded) */
struct ResultSet {
    size_t k;
    std::set<Pair, PairLess> s;
    /* adds to a full set whose distance equals the last entry's: the reference keeps the older entry whatever the
     * ids, where a selection of the k smallest (distance, id) keys may keep the newer one. Counted so that tests can
     * tell an exact distance tie from a real difference. */
    size_t ties = 0;
    explicit ResultSet(size_t k_) : k(k_) {}
    bool add(Pair p) { /* :61-74 */
        if (s.size() < k) {
            s.insert(p);
            return true;
        }
        if (!s.empty()) {
            auto last = std::prev(s.end());
            const int c = cmp_of(p.d, last->d);
            if (c < 0) { /* strict, distance only */
                s.erase(last);
                s.insert(p);
                return true;
            }
            if (c == 0) ++ties;
        }
        return false;
    }
};

size_t emit(const ResultSet& rs, size_t k, uint64_t* ids, float* dd) {
    size_t c = 0;
    for (const Pair& p : rs.s) {
        if (c >= k) break;
        ids[c] = p.i;
        dd[c] = p.d;
        ++c;
    }
    for (size_t j = c; j < k; ++j) {
        ids[j] = UINT64_MAX;
        dd[j] = std::numeric_limits<float>::quiet_NaN();
    }
    return c;
}

template <class F> void parallel_for(size_t n, int nthreads, F f) {
    if (nthreads <= 1 || n <= 1) {
        for (size_t i = 0; i < n; ++i) f(i);
        return;
    }
    std::atomic<size_t> next(0);
    std::vector<std::thread> th;
    size_t nt = std::min<size_t>(nthreads, n);
    for (size_t t = 0; t < nt; ++t)
        th.emplace_back([&] {
            for (;;) {
                size_t i = next.fetch_add(1);
                if (i >= n) break;
                f(i);
            }
        });
    for (auto& t : th) t.join();
}
/* chunked variant for cheap per-item work */
template <class F> void parallel_chunks(size_t n, int nthreads, size_t chunk, F f) {
    size_t nchunks = (n + chunk - 1) / chunk;
    parallel_for(nchunks, nthreads, [&](size_t c) {
        size_t lo = c * chunk, hi = std::min(n, lo + chunk);
        for (size_t i = lo; i < hi; ++i) f(i);
    });
}

/* ---- flat_index.rs:48-57 ---------------------------------------------------------------- */
template <class T>
void flat_knn_one(const T* base, size_t n, size_t dim, int metric, const T* q, size_t k,
                  uint64_t* ids, float* dd, uint32_t* count) {
    ResultSet rs(k);
    for (size_t i = 0; i < n; ++i) rs.add({dist(q, base + i * dim, dim, metric), i});
    *count = (uint32_t)emit(rs, k, ids, dd);
}

/* ---- k_means.rs:40-57: argmin by (distance, index) --------------------------------------- */
template <class T>
uint64_t find_nearest_base(const T* v, const T* cent, size_t k, size_t d, int metric) {
    Pair best{0.0f, 0};
    PairLess less;
    for (size_t c = 0; c < k; ++c) {
        Pair p{dist(v, cent + c * d, d, metric), c};
        if (c == 0 || less(p, best)) best = p;
    }
    return best.i;
}

/* ---- pq_table.rs:38-53 ------------------------------------------------------------------- */
std::vector<std::pair<size_t, size_t>> pq_groups(size_t dim, size_t m) {
    std::vector<std::pair<size_t, size_t>> g;
    size_t cur = 0;
    while (cur < dim) {
        size_t rem = m - g.size();
        size_t gs = (dim - cur + rem - 1) / rem;
        g.emplace_back(cur, cur + gs);
        cur += gs;
    }
    return g;
}

/* ---- pq_table.rs:66-91 ------------------------------------------------------------------- */
template <class T>
void pq_encode_one(const T* v, size_t dim, int metric, const T* codebooks, size_t m, size_t n_bits,
                   const std::vector<std::pair<size_t, size_t>>& groups,
                   const std::vector<size_t>& cb_off, uint8_t* out) {
    size_t kc = (size_t)1 << n_bits;
    auto nearest = [&](size_t g) {
        size_t lo = groups[g].first, hi = groups[g].second;
        return find_nearest_base(v + lo, codebooks + cb_off[g], kc, hi - lo, metric);
    };
    (void)dim;
    if (n_bits == 4) {
        size_t enc = (m + 1) / 2;
        std::memset(out, 0, enc);
        for (size_t i = 0; i < m / 2; ++i) {
            uint64_t v0 = nearest(2 * i), v1 = nearest(2 * i + 1);
            out[i] = (uint8_t)(v0 | (v1 << 4));
        }
        if (m % 2 == 1) out[m / 2] = (uint8_t)nearest(m - 1);
    } else {
        for (size_t g = 0; g < m; ++g) out[g] = (uint8_t)nearest(g);
    }
}

std::vector<size_t> codebook_offsets(const std::vector<std::pair<size_t, size_t>>& groups, size_t kc) {
    std::vector<size_t> off(groups.size() + 1, 0);
    for (size_t g = 0; g < groups.size(); ++g)
        off[g + 1] = off[g] + kc * (groups[g].second - groups[g].first);
    return off;
}

/* ---- pq_table.rs:239-301 ----------------------------------------------------------------- */
float pq_adc(const uint8_t* code, size_t m, size_t n_bits, int metric, const float* lut,
             const float* dist_cache, float qcache) {
    size_t kc = (size_t)1 << n_bits;
    float sum = 0.0f, cdp = 0.0f;
    auto push_one = [&](size_t i, size_t idx) {
        if (i >= m) return;
        sum = sum + lut[i * kc + idx];
        if (metric == ORC_COSINE) cdp = cdp + dist_cache[i * kc + idx];
    };
    if (n_bits == 4) {
        size_t enc = (m + 1) / 2, i = 0;
        for (size_t b = 0; b < enc; ++b) {
            push_one(i++, code[b] & 0xf);
            push_one(i++, code[b] >> 4);
        }
    } else {
        for (size_t i = 0; i < m; ++i) push_one(i, code[i]);
    }
    if (metric == ORC_L2SQR) return sum;
    float norm0 = std::sqrt(cdp);
    float den = rmax(norm0 * qcache, 1e-10f);
    float q = sum / den;
    return 1.0f - q;
}

/* ---- pq_table.rs:195-224 ----------------------------------------------------------------- */
template <class T>
void pq_lookup(const T* q, size_t dim, int metric, const T* codebooks, size_t m, size_t n_bits,
               float* lut, float* qcache) {
    size_t kc = (size_t)1 << n_bits;
    auto groups = pq_groups(dim, m);
    auto off = codebook_offsets(groups, kc);
    for (size_t g = 0; g < groups.size(); ++g) {
        size_t lo = groups[g].first, d = groups[g].second - lo;
        for (size_t c = 0; c < kc; ++c) {
            const T* cc = codebooks + off[g] + c * d;
            lut[g * kc + c] = metric == ORC_L2SQR ? l2sqr(q + lo, cc, d) : dot(q + lo, cc, d);
        }
    }
    *qcache = metric == ORC_L2SQR ? 0.0f : vec_norm(q, dim);
}
template <class T>
void pq_dist_cache(size_t dim, int metric, const T* codebooks, size_t m, size_t n_bits, float* out) {
    size_t kc = (size_t)1 << n_bits;
    auto groups = pq_groups(dim, m);
    auto off = codebook_offsets(groups, kc);
    for (size_t g = 0; g < groups.size(); ++g) {
        size_t d = groups[g].second - groups[g].first;
        for (size_t c = 0; c < kc; ++c) {
            const T* cc = codebooks + off[g] + c * d;
            out[g * kc + c] = metric == ORC_L2SQR ? 0.0f : dot(cc, cc, d);
        }
    }
}

void adc_topk(size_t n, int metric, const uint8_t* codes, size_t m, size_t n_bits, const float* lut,
              const float* dist_cache, float qcache, size_t kk, ResultSet& rs) {
    size_t enc = n_bits == 4 ? (m + 1) / 2 : m;
    (void)kk;
    for (size_t i = 0; i < n; ++i)
        rs.add({pq_adc(codes + i * enc, m, n_bits, metric, lut, dist_cache, qcache), i});
}

/* ---- flat_index.rs:84-104 + candidate_pair.rs:102-108 -------------------------------------- */
template <class T>
void flat_knn_pq_one(const T* base, size_t n, size_t dim, int metric, const uint8_t* codes,
                     const T* codebooks, const float* dist_cache, size_t m, size_t n_bits, const T* q,
                     size_t k, size_t ef, uint64_t* ids, float* dd, uint32_t* count) {
    size_t kc = (size_t)1 << n_bits;
    std::vector<float> lut(m * kc);
    float qcache;
    pq_lookup(q, dim, metric, codebooks, m, n_bits, lut.data(), &qcache);
    ResultSet pq(std::max(ef, k));
    adc_topk(n, metric, codes, m, n_bits, lut.data(), dist_cache, qcache, std::max(ef, k), pq);
    ResultSet rs(k); /* pq_resort: iterate ascending (adc, index) */
    for (const Pair& p : pq.s) rs.add({dist(q, base + p.i * dim, dim, metric), p.i});
    *count = (uint32_t)emit(rs, k, ids, dd);
}

/* ---- k_means.rs:174-191 -------------------------------------------------------------------- */
template <class T>
size_t find_n_nearest(const T* v, const T* cent, size_t k, size_t dim, int metric, size_t n_probes,
                      uint64_t* out) {
    ResultSet rs(n_probes);
    for (size_t c = 0; c < k; ++c) rs.add({dist(v, cent + c * dim, dim, metric), c});
    size_t j = 0;
    for (const Pair& p : rs.s) out[j++] = p.i;
    return j;
}

/* ---- ivf_index.rs:143-154 ------------------------------------------------------------------ */
template <class T>
void ivf_knn_one(const T* base, size_t dim, int metric, const T* cent, size_t nlist,
                 const uint64_t* offsets, const uint64_t* members, const T* q, size_t k,
                 size_t n_probes, uint64_t* ids, float* dd, uint32_t* count) {
    std::vector<uint64_t> probes(std::min(n_probes, nlist));
    size_t np = find_n_nearest(q, cent, nlist, dim, metric, n_probes, probes.data());
    ResultSet rs(k);
    for (size_t p = 0; p < np; ++p) {
        uint64_t c = probes[p];
        for (uint64_t j = offsets[c]; j < offsets[c + 1]; ++j) {
            uint64_t i = members[j];
            rs.add({dist(base + i * dim, q, dim, metric), i}); /* d(v, query), ivf_index.rs:150 */
        }
    }
    *count = (uint32_t)emit(rs, k, ids, dd);
}

/* ---- k_means.rs:108-161: Lloyd ------------------------------------------------------------- */
template <class T>
int lloyd(const T* rows, size_t n, size_t dim, int metric, T* cent, size_t k, size_t lo, size_t hi,
          size_t max_iter, float tol, int nthreads) {
    size_t d = hi - lo;
    std::vector<float> sums(k * d, 0.0f);
    std::vector<uint32_t> assign(n);
    std::vector<T> newc(k * d);
    int iters = 0;
    for (size_t it = 0; it < max_iter; ++it) {
        ++iters;
        parallel_chunks(n, nthreads, 256, [&](size_t i) {
            assign[i] = (uint32_t)find_nearest_base(rows + i * dim + lo, cent, k, d, metric);
        });
        std::vector<std::vector<size_t>> members(k);
        for (size_t i = 0; i < n; ++i) members[assign[i]].push_back(i);
        for (size_t c = 0; c < k; ++c) {
            float* s = sums.data() + c * d;
            if (members[c].empty()) { /* :131-137 keep unchanged */
                for (size_t j = 0; j < d; ++j) s[j] = to_f32(cent[c * d + j]);
                continue;
            }
            for (size_t j = 0; j < d; ++j) s[j] = 0.0f;
            for (size_t i : members[c]) { /* ascending member order, f32 sums */
                const T* v = rows + i * dim + lo;
                for (size_t j = 0; j < d; ++j) s[j] = s[j] + to_f32(v[j]);
            }
            float cnt = (float)members[c].size();
            for (size_t j = 0; j < d; ++j) s[j] = s[j] / cnt;
        }
        for (size_t j = 0; j < k * d; ++j) newc[j] = from_f32<T>(sums[j]); /* to_type :149 */
        float max_diff = -std::numeric_limits<float>::infinity();
        for (size_t c = 0; c < k; ++c)
            max_diff = rmax(max_diff, l2sqr(cent + c * d, newc.data() + c * d, d));
        std::memcpy(cent, newc.data(), k * d * sizeof(T));
        if (max_diff < tol) break;
    }
    return iters;
}

/* splitmix64: the ORACLE'S OWN rng (the reference's ChaCha12 stream is not restated) */
struct SplitMix {
    uint64_t s;
    uint64_t next() {
        uint64_t z = (s += 0x9E3779B97F4A7C15ull);
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        return z ^ (z >> 31);
    }
    double uniform() { return (double)(next() >> 11) * (1.0 / 9007199254740992.0); }
    size_t below(size_t n) { return (size_t)(uniform() * (double)n) % n; }
};

/* ---- k_means.rs:75-77: the k-means++ weight update w[i] = min(w[i], d(c, v_i[lo:hi])) -------- */
template <class T>
void kmeans_pp_weights(const T* rows, size_t n, size_t dim, int metric, const T* c, size_t lo, size_t hi, float* w,
                       int nthreads) {
    parallel_chunks(n, nthreads, 256, [&](size_t i) {
        w[i] = std::fmin(w[i], dist(c, rows + i * dim + lo, hi - lo, metric)); /* d(c, v) :76, f32::min */
    });
}

/* ---- k_means.rs:61-87: k-means++ (structure only; draws are not the reference's) ----------- */
template <class T>
void kmeans_pp(const T* rows, size_t n, size_t dim, int metric, size_t k, size_t lo, size_t hi,
               uint64_t seed, T* cent) {
    size_t d = hi - lo;
    SplitMix rng{seed};
    size_t first = rng.below(n);
    std::memcpy(cent, rows + first * dim + lo, d * sizeof(T));
    std::vector<float> w(n, std::numeric_limits<float>::infinity());
    for (size_t idx = 1; idx < k; ++idx) {
        kmeans_pp_weights(rows, n, dim, metric, cent + (idx - 1) * d, lo, hi, w.data(), 1);
        double total = 0.0;
        bool ok = true;
        for (size_t i = 0; i < n; ++i) {
            if (!(w[i] >= 0.0f) || std::isinf(w[i])) ok = false; /* WeightedIndex rejects <0 / NaN */
            total += w[i];
        }
        size_t fallback = rng.below(n); /* eager unwrap_or argument :80-82 */
        size_t c = fallback;
        if (ok && total > 0.0) {
            double r = rng.uniform() * total, acc = 0.0;
            c = n - 1;
            for (size_t i = 0; i < n; ++i) {
                acc += w[i];
                if (r < acc) {
                    c = i;
                    break;
                }
            }
        }
        std::memcpy(cent + idx * d, rows + c * dim + lo, d * sizeof(T));
    }
}

}  // namespace

#define DISPATCH(dtype, expr_f32, expr_u8)   \
    do {                                     \
        if ((dtype) == ORC_F32) {            \
            typedef float T;                 \
            expr_f32;                        \
        } else {                             \
            typedef uint8_t T;               \
            expr_u8;                         \
        }                                    \
    } while (0)
#define D1(dtype, expr) DISPATCH(dtype, expr, expr)


/* ---- hnsw_index.rs: HNSWIndex restated for one thread (add :538-572 for every row, i.e. the reference's own path
 * while len < start_batch_since and whenever it is given one vector at a time; knn_with_ef :616-625). The graph of
 * the reference is RNG- and thread-count dependent, so this is a recall yardstick, not a golden graph. ---- */
template <class T> struct Hnsw {
    const T* rows;
    size_t n = 0, dim, m, max_m0, ef_c;
    int metric;
    std::vector<uint32_t> level0;            /* [n][max_m0] */
    std::vector<std::vector<uint32_t>> other; /* [n][level * m] */
    std::vector<std::vector<size_t>> len;     /* [n][level + 1] */
    std::vector<size_t> vec_level;
    std::vector<float> cache;
    long enter_level = -1, enter_point = -1;

    size_t limit(size_t level) const { return level == 0 ? max_m0 : m; }
    const uint32_t* links(size_t v, size_t level) const {
        return level == 0 ? &level0[v * max_m0] : &other[v][m * (level - 1)];
    }
    uint32_t* links(size_t v, size_t level) { return level == 0 ? &level0[v * max_m0] : &other[v][m * (level - 1)]; }
    float d_cached(size_t idx, const T* q, float qc) const { /* dist_with_cache :351-355 */
        const T* v = rows + idx * dim;
        return metric == ORC_L2SQR ? l2sqr_cached(v, q, dim, cache[idx], qc) : cosine_cached(v, q, dim, cache[idx], qc);
    }
    float inner(size_t a, size_t b) const { return d_cached(a, rows + b * dim, cache[b]); } /* :356-358 */
    template <class F> ResultSet search_on_level(size_t enter, size_t level, size_t ef, F dist_fn) const { /* :258-291 */
        std::set<size_t> visited;
        std::set<Pair, PairLess> queue;
        ResultSet result(ef);
        visited.insert(enter);
        Pair ep{dist_fn(enter), enter};
        result.add(ep);
        queue.insert(ep);
        while (!queue.empty()) {
            Pair p = *queue.begin();
            queue.erase(queue.begin());
            /* check_candidate :55-57 */
            if (!(result.s.size() < result.k || PairLess()(p, *std::prev(result.s.end())))) break;
            const uint32_t* lk = links(p.i, level);
            for (size_t j = 0; j < len[p.i][level]; ++j) {
                size_t nb = lk[j];
                if (!visited.insert(nb).second) continue;
                Pair np{dist_fn(nb), nb};
                result.add(np);
                queue.insert(np);
            }
        }
        return result;
    }
    template <class F> size_t greedy(size_t target, F dist_fn) const { /* :306-350 */
        size_t level = (size_t)enter_level, cur = (size_t)enter_point;
        while (level > target) {
            float cur_d = dist_fn(cur);
            for (;;) {
                bool flag = false;
                size_t at = cur;
                const uint32_t* lk = links(at, level);
                for (size_t j = 0; j < len[at][level]; ++j) {
                    float nd = dist_fn(lk[j]);
                    if (nd < cur_d) {
                        cur_d = nd;
                        cur = lk[j];
                        flag = true;
                    }
                }
                if (!flag) break;
            }
            --level;
        }
        return cur;
    }
    std::vector<Pair> heuristic(const std::set<Pair, PairLess>& cand, size_t mm) const { /* candidate_pair.rs:85-99 */
        std::vector<Pair> nb;
        for (const Pair& p : cand) {
            if (nb.size() >= mm) break;
            bool ok = true;
            for (const Pair& r : nb)
                if (!(inner(p.i, r.i) >= p.d)) {
                    ok = false;
                    break;
                }
            if (ok) nb.push_back(p);
        }
        return nb;
    }
    void arrange(size_t v, size_t level, size_t nv) { /* :204-224 */
        size_t lim = limit(level);
        std::vector<uint32_t> lk(links(v, level), links(v, level) + len[v][level]);
        lk.push_back((uint32_t)nv);
        if (lk.size() > lim) {
            ResultSet set(lim + 1);
            for (uint32_t x : lk) set.add(Pair{inner(v, x), x});
            auto keep = heuristic(set.s, lim);
            lk.clear();
            for (const Pair& p : keep) lk.push_back((uint32_t)p.i);
        }
        len[v][level] = lk.size();
        std::copy(lk.begin(), lk.end(), links(v, level));
    }
    uint64_t build_ties = 0; /* tie events (ResultSet::ties) of every candidate search of the build */
    void push_init(size_t idx, size_t level) { /* :241-256: a node without links */
        level0.resize((idx + 1) * max_m0, 0);
        other.emplace_back(m * level, 0u);
        len.emplace_back(level + 1, (size_t)0);
        vec_level.push_back(level);
        const T* v = rows + idx * dim;
        cache.push_back(metric == ORC_L2SQR ? dot(v, v, dim) : vec_norm(v, dim));
        n = idx + 1;
    }
    void add(size_t idx, size_t level) { /* push_init :241-256 + add :538-572 */
        push_init(idx, level);
        if (enter_point < 0) {
            enter_level = (long)level;
            enter_point = (long)idx;
            return;
        }
        const T* v = rows + idx * dim;
        const float qc = cache[idx];
        auto dist_fn = [&](size_t i) { return d_cached(i, v, qc); };
        size_t cur = (long)level < enter_level ? greedy(level, dist_fn) : (size_t)enter_point;
        for (long l = std::min<long>((long)level, enter_level); l >= 0; --l) {
            ResultSet cand = search_on_level(cur, (size_t)l, ef_c, dist_fn);
            build_ties += cand.ties;
            cur = cand.s.begin()->i;
            auto nb = heuristic(cand.s, m); /* connect_new_links :226-239 */
            for (size_t j = 0; j < nb.size(); ++j) links(idx, (size_t)l)[j] = (uint32_t)nb[j].i;
            len[idx][(size_t)l] = nb.size();
            for (const Pair& p : nb) arrange(p.i, (size_t)l, idx);
        }
        if ((long)level > enter_level) {
            enter_level = (long)level;
            enter_point = (long)idx;
        }
    }
    /* The device build (hnsw.cu, hnsw_insert_range) restated: rows [n, end) are inserted a batch at a time, batch
     * size min(max(1, done / m), max_batch, rows left). Every node of a batch searches the graph as it stood when the
     * batch began; on each level the entry of the next level is the graph search's best, taken before the candidates
     * are merged with the earlier nodes of the batch that live on that level. Then every (node, level) selects its
     * links (at most m, level 0 too), then the back-links are applied grouped by (level, target), the sources of a
     * target in task order (node, then level upwards). The enter point moves after the batch. With max_batch = 1 this
     * is `add` row by row. */
    void insert_batched(size_t end, const uint32_t* levels, size_t max_batch) {
        size_t done = n;
        if (done >= end) return;
        if (enter_point < 0) { /* the first vector becomes the enter point (:543-551) */
            add(done, levels[done]);
            ++done;
        }
        while (done < end) {
            const size_t b = std::min(std::min(std::max<size_t>(1, done / m), max_batch), end - done);
            const size_t first = done;
            for (size_t i = first; i < first + b; ++i) push_init(i, levels[i]);
            struct Task {
                size_t node, level;
                std::vector<Pair> sel;
            };
            std::vector<Task> tasks;
            std::vector<std::vector<ResultSet>> cands(b); /* [node][level] */
            for (size_t i = first; i < first + b; ++i) {
                const T* v = rows + i * dim;
                const float qc = cache[i];
                auto dist_fn = [&](size_t x) { return d_cached(x, v, qc); };
                const size_t level = levels[i];
                size_t cur = (long)level < enter_level ? greedy(level, dist_fn) : (size_t)enter_point;
                const long top = std::min<long>((long)level, enter_level);
                cands[i - first].assign((size_t)top + 1, ResultSet(0));
                for (long l = top; l >= 0; --l) {
                    ResultSet cand = search_on_level(cur, (size_t)l, ef_c, dist_fn);
                    cur = cand.s.begin()->i;
                    for (size_t j = first; j < i; ++j) /* brute force among the batch (:431-437) */
                        if ((long)levels[j] >= l) cand.add(Pair{dist_fn(j), j});
                    build_ties += cand.ties;
                    cands[i - first][(size_t)l] = std::move(cand);
                }
            }
            for (size_t i = first; i < first + b; ++i)
                for (size_t l = 0; l < cands[i - first].size(); ++l) {
                    Task t{i, l, heuristic(cands[i - first][l].s, m)};
                    for (size_t j = 0; j < t.sel.size(); ++j) links(i, l)[j] = (uint32_t)t.sel[j].i;
                    len[i][l] = t.sel.size();
                    tasks.push_back(std::move(t));
                }
            struct Back {
                size_t level, target, source;
            };
            std::vector<Back> back;
            for (const Task& t : tasks)
                for (const Pair& p : t.sel) back.push_back(Back{t.level, p.i, t.node});
            std::stable_sort(back.begin(), back.end(), [](const Back& a, const Back& c) {
                return a.level != c.level ? a.level < c.level : a.target < c.target;
            });
            for (const Back& e : back) arrange(e.target, e.level, e.source);
            for (size_t i = first; i < first + b; ++i)
                if ((long)levels[i] > enter_level) {
                    enter_level = (long)levels[i];
                    enter_point = (long)i;
                }
            done += b;
        }
    }
};

extern "C" {

float orc_dot(const void* a, const void* b, size_t dim, int dtype) {
    D1(dtype, return dot((const T*)a, (const T*)b, dim));
    return 0;
}
float orc_l2_sqr(const void* a, const void* b, size_t dim, int dtype) {
    D1(dtype, return l2sqr((const T*)a, (const T*)b, dim));
    return 0;
}
float orc_vec_norm(const void* a, size_t dim, int dtype) {
    D1(dtype, return vec_norm((const T*)a, dim));
    return 0;
}
float orc_distance(const void* a, const void* b, size_t dim, int dtype, int metric) {
    D1(dtype, return dist((const T*)a, (const T*)b, dim, metric));
    return 0;
}
float orc_distance_cached(const void* a, const void* b, size_t dim, int dtype, int metric,
                          float ca, float cb) {
    D1(dtype, return metric == ORC_L2SQR ? l2sqr_cached((const T*)a, (const T*)b, dim, ca, cb)
                                         : cosine_cached((const T*)a, (const T*)b, dim, ca, cb));
    return 0;
}
float orc_dist_cache(const void* a, size_t dim, int dtype, int metric) {
    D1(dtype, return metric == ORC_L2SQR ? dot((const T*)a, (const T*)a, dim)
                                         : vec_norm((const T*)a, dim));
    return 0;
}

int orc_flat_knn(const void* base, size_t n, size_t dim, int dtype, int metric, const void* queries,
                 size_t nq, size_t k, uint64_t* ids, float* dd, uint32_t* counts, int nthreads) {
    D1(dtype, parallel_for(nq, nthreads, [&](size_t q) {
           flat_knn_one((const T*)base, n, dim, metric, (const T*)queries + q * dim, k, ids + q * k,
                        dd + q * k, counts + q);
       }));
    return 0;
}

int orc_pq_groups(size_t dim, size_t m, uint64_t* out) {
    if (dim == 0 || m == 0 || dim < m) return 1;
    auto g = pq_groups(dim, m);
    for (size_t i = 0; i < g.size(); ++i) {
        out[2 * i] = g[i].first;
        out[2 * i + 1] = g[i].second;
    }
    return 0;
}

uint64_t orc_find_nearest(const void* v, const void* centroids, size_t k, size_t sel_lo,
                          size_t sel_hi, int dtype, int metric) {
    D1(dtype, return find_nearest_base((const T*)v + sel_lo, (const T*)centroids, k, sel_hi - sel_lo,
                                       metric));
    return 0;
}
size_t orc_find_n_nearest(const void* v, const void* centroids, size_t k, size_t dim, int dtype,
                          int metric, size_t n_probes, uint64_t* out) {
    D1(dtype, return find_n_nearest((const T*)v, (const T*)centroids, k, dim, metric, n_probes, out));
    return 0;
}
int orc_kmeans_assign(const void* rows, size_t n, size_t dim, int dtype, int metric,
                      const void* centroids, size_t k, size_t sel_lo, size_t sel_hi, uint32_t* out,
                      int nthreads) {
    D1(dtype, parallel_chunks(n, nthreads, 256, [&](size_t i) {
           out[i] = (uint32_t)find_nearest_base((const T*)rows + i * dim + sel_lo, (const T*)centroids,
                                                k, sel_hi - sel_lo, metric);
       }));
    return 0;
}
int orc_kmeans_lloyd(const void* rows, size_t n, size_t dim, int dtype, int metric, void* centroids,
                     size_t k, size_t sel_lo, size_t sel_hi, size_t max_iter, float tol) {
    D1(dtype, return lloyd((const T*)rows, n, dim, metric, (T*)centroids, k, sel_lo, sel_hi, max_iter,
                           tol, (int)std::max(1u, std::thread::hardware_concurrency())));
    return 0;
}
int orc_kmeans_pp_init(const void* rows, size_t n, size_t dim, int dtype, int metric, size_t k,
                       size_t sel_lo, size_t sel_hi, uint64_t seed, void* centroids) {
    if (n == 0 || k == 0) return 1;
    D1(dtype, kmeans_pp((const T*)rows, n, dim, metric, k, sel_lo, sel_hi, seed, (T*)centroids));
    return 0;
}
int orc_kmeans_pp_weights(const void* rows, size_t n, size_t dim, int dtype, int metric, const void* c, size_t sel_lo,
                          size_t sel_hi, float* w, int nthreads) {
    if (sel_lo > sel_hi || sel_hi > dim) return 1;
    D1(dtype, kmeans_pp_weights((const T*)rows, n, dim, metric, (const T*)c, sel_lo, sel_hi, w, nthreads));
    return 0;
}

int orc_pq_encode(const void* rows, size_t n, size_t dim, int dtype, int metric, const void* codebooks,
                  size_t m, size_t n_bits, uint8_t* codes, int nthreads) {
    if (n_bits != 4 && n_bits != 8) return 1;
    size_t kc = (size_t)1 << n_bits;
    auto groups = pq_groups(dim, m);
    auto off = codebook_offsets(groups, kc);
    size_t enc = n_bits == 4 ? (m + 1) / 2 : m;
    D1(dtype, parallel_chunks(n, nthreads, 64, [&](size_t i) {
           pq_encode_one((const T*)rows + i * dim, dim, metric, (const T*)codebooks, m, n_bits, groups,
                         off, codes + i * enc);
       }));
    return 0;
}
int orc_pq_lookup(const void* q, size_t dim, int dtype, int metric, const void* codebooks, size_t m,
                  size_t n_bits, float* lut, float* qcache) {
    D1(dtype, pq_lookup((const T*)q, dim, metric, (const T*)codebooks, m, n_bits, lut, qcache));
    return 0;
}
int orc_pq_dist_cache(size_t dim, int dtype, int metric, const void* codebooks, size_t m,
                      size_t n_bits, float* out) {
    D1(dtype, pq_dist_cache(dim, metric, (const T*)codebooks, m, n_bits, out));
    return 0;
}
float orc_pq_adc(const uint8_t* code, size_t m, size_t n_bits, int metric, const float* lut,
                 const float* dist_cache, float qcache) {
    return pq_adc(code, m, n_bits, metric, lut, dist_cache, qcache);
}
int orc_flat_knn_pq(const void* base, size_t n, size_t dim, int dtype, int metric,
                    const uint8_t* codes, const void* codebooks, size_t m, size_t n_bits,
                    const void* queries, size_t nq, size_t k, size_t ef, uint64_t* ids, float* dd,
                    uint32_t* counts, int nthreads) {
    size_t kc = (size_t)1 << n_bits;
    std::vector<float> dcache(m * kc);
    orc_pq_dist_cache(dim, dtype, metric, codebooks, m, n_bits, dcache.data());
    D1(dtype, parallel_for(nq, nthreads, [&](size_t q) {
           flat_knn_pq_one((const T*)base, n, dim, metric, codes, (const T*)codebooks, dcache.data(), m,
                           n_bits, (const T*)queries + q * dim, k, ef, ids + q * k, dd + q * k,
                           counts + q);
       }));
    return 0;
}
int orc_flat_adc_topk(size_t n, int metric, const uint8_t* codes, size_t m, size_t n_bits,
                      const float* lut, const float* dist_cache, float qcache, size_t kk,
                      uint64_t* ids, float* dd, uint32_t* count) {
    ResultSet rs(kk);
    adc_topk(n, metric, codes, m, n_bits, lut, dist_cache, qcache, kk, rs);
    *count = (uint32_t)emit(rs, kk, ids, dd);
    return 0;
}

int orc_ivf_lists(const uint32_t* assign, size_t n, size_t nlist, uint64_t* offsets,
                  uint64_t* members) {
    std::vector<uint64_t> cnt(nlist + 1, 0);
    for (size_t i = 0; i < n; ++i) {
        if (assign[i] >= nlist) return 1;
        cnt[assign[i] + 1]++;
    }
    offsets[0] = 0;
    for (size_t c = 0; c < nlist; ++c) offsets[c + 1] = offsets[c] + cnt[c + 1];
    std::vector<uint64_t> pos(offsets, offsets + nlist);
    for (size_t i = 0; i < n; ++i) members[pos[assign[i]]++] = i; /* ascending inside a list */
    return 0;
}
int orc_ivf_knn(const void* base, size_t n, size_t dim, int dtype, int metric, const void* centroids,
                size_t nlist, const uint64_t* offsets, const uint64_t* members, const void* queries,
                size_t nq, size_t k, size_t n_probes, uint64_t* ids, float* dd, uint32_t* counts,
                int nthreads) {
    (void)n;
    if (n_probes == 0) return 1; /* assert k_means.rs:175-178 */
    D1(dtype, parallel_for(nq, nthreads, [&](size_t q) {
           ivf_knn_one((const T*)base, dim, metric, (const T*)centroids, nlist, offsets, members,
                       (const T*)queries + q * dim, k, n_probes, ids + q * k, dd + q * k, counts + q);
       }));
    return 0;
}

int orc_gather_dist(const void* base, size_t dim, int dtype, int metric, const float* row_cache,
                    const void* query, float query_cache, const uint64_t* cand, size_t ncand,
                    float* out) {
    D1(dtype, for (size_t j = 0; j < ncand; ++j) {
        const T* v = (const T*)base + cand[j] * dim;
        out[j] = metric == ORC_L2SQR
                     ? l2sqr_cached((const T*)query, v, dim, query_cache, row_cache[cand[j]])
                     : cosine_cached((const T*)query, v, dim, query_cache, row_cache[cand[j]]);
    });
    return 0;
}


/* HNSW handle (f32 / u8 rows are borrowed: the caller keeps `rows` alive) */
void* orc_hnsw_build(const void* rows, size_t n, size_t dim, int dtype, int metric, size_t m, size_t ef_construction,
                     const uint32_t* levels) {
    D1(dtype, {
        auto* h = new Hnsw<T>();
        h->rows = (const T*)rows;
        h->dim = dim;
        h->m = m;
        h->max_m0 = 2 * m;                                   /* :503 */
        h->ef_c = std::max(ef_construction, 2 * m);          /* :504 */
        h->metric = metric;
        for (size_t i = 0; i < n; ++i) h->add(i, levels[i]);
        return (void*)h;
    });
    return nullptr;
}
/* The device build's batch pipeline (Hnsw::insert_batched): rows [0, n0) are inserted as one build, then rows [n0, n)
 * as an append onto that graph (batch sizes restart from done = n0, like vdb_hnsw_append). n0 = 0: one build. */
void* orc_hnsw_build_batched(const void* rows, size_t n, size_t dim, int dtype, int metric, size_t m, size_t ef_construction,
                             const uint32_t* levels, size_t max_batch, size_t n0) {
    if (max_batch == 0 || n0 > n) return nullptr;
    D1(dtype, {
        auto* h = new Hnsw<T>();
        h->rows = (const T*)rows;
        h->dim = dim;
        h->m = m;
        h->max_m0 = 2 * m;
        h->ef_c = std::max(ef_construction, 2 * m);
        h->metric = metric;
        h->insert_batched(n0, levels, max_batch);
        h->insert_batched(n, levels, max_batch);
        return (void*)h;
    });
    return nullptr;
}
uint64_t orc_hnsw_build_ties(const void* handle, int dtype) {
    D1(dtype, return ((const Hnsw<T>*)handle)->build_ties);
    return 0;
}
int orc_hnsw_enter(const void* handle, int dtype, long* enter_point, long* enter_level) {
    D1(dtype, {
        *enter_point = ((const Hnsw<T>*)handle)->enter_point;
        *enter_level = ((const Hnsw<T>*)handle)->enter_level;
    });
    return 0;
}
/* An index whose graph was built elsewhere (HNSWIndex deserialisation, hnsw_index.rs:641-668, followed by
 * init_dist_cache_after_load :371-379): levels[n], level-0 links [n][2m] + lengths, upper levels per node in row order
 * ([sum(levels)][m] + lengths). Lets the CPU search walk the very graph the GPU built. */
void* orc_hnsw_from_graph(const void* rows, size_t n, size_t dim, int dtype, int metric, size_t m, size_t ef_construction,
                          const uint32_t* levels, const uint32_t* links0, const uint32_t* len0, const uint32_t* ulinks,
                          const uint32_t* ulen, long enter_point, long enter_level) {
    D1(dtype, {
        auto* h = new Hnsw<T>();
        h->rows = (const T*)rows;
        h->n = n;
        h->dim = dim;
        h->m = m;
        h->max_m0 = 2 * m;
        h->ef_c = std::max(ef_construction, 2 * m);
        h->metric = metric;
        h->level0.assign(links0, links0 + n * h->max_m0);
        h->other.resize(n);
        h->len.resize(n);
        h->vec_level.resize(n);
        h->cache.resize(n);
        size_t slot = 0;
        for (size_t i = 0; i < n; ++i) {
            const size_t lv = levels[i];
            h->vec_level[i] = lv;
            h->len[i].assign(lv + 1, 0);
            h->len[i][0] = len0[i];
            h->other[i].assign(lv * m, 0);
            for (size_t l = 1; l <= lv; ++l, ++slot) {
                h->len[i][l] = ulen[slot];
                std::copy(ulinks + slot * m, ulinks + (slot + 1) * m, h->other[i].begin() + (l - 1) * m);
            }
            const T* v = h->rows + i * dim;
            h->cache[i] = metric == ORC_L2SQR ? dot(v, v, dim) : vec_norm(v, dim);   /* dist_cache, distance/mod.rs:31-36 */
        }
        h->enter_point = enter_point;
        h->enter_level = enter_level;
        return (void*)h;
    });
    return nullptr;
}
int orc_hnsw_knn(const void* handle, int dtype, const void* queries, size_t nq, size_t k, size_t ef, uint64_t* ids,
                 float* dists, uint32_t* counts, int nthreads, uint32_t* ties) {
    D1(dtype, {
        const auto* h = (const Hnsw<T>*)handle;
        parallel_for(nq, nthreads, [&](size_t q) {
            const T* qv = (const T*)queries + q * h->dim;
            if (ties) ties[q] = 0;
            if (h->n == 0) {
                counts[q] = 0;
                return;
            }
            const float qc = h->metric == ORC_L2SQR ? dot(qv, qv, h->dim) : vec_norm(qv, h->dim);
            auto dist_fn = [&](size_t i) { return h->d_cached(i, qv, qc); };
            size_t ep = h->greedy(0, dist_fn);
            ResultSet r = h->search_on_level(ep, 0, std::max(ef, k), dist_fn);
            counts[q] = (uint32_t)emit(r, k, ids + q * k, dists + q * k);
            if (ties) ties[q] = (uint32_t)r.ties;
        });
    });
    return 0;
}
/* HNSWIndex::knn_pq (hnsw_index.rs:672-697): graph walk with ADC distances, then pq_resort with dist_with_cache */
int orc_hnsw_knn_pq(const void* handle, int dtype, const void* queries, size_t nq, size_t k, size_t ef, const uint8_t* codes,
                    const void* codebooks, size_t m, size_t n_bits, uint64_t* ids, float* dists, uint32_t* counts, int nthreads,
                    uint32_t* ties) {
    D1(dtype, {
        const auto* h = (const Hnsw<T>*)handle;
        const size_t kc = (size_t)1 << n_bits;
        const size_t enc = n_bits == 4 ? (m + 1) / 2 : m;
        std::vector<float> dcache(m * kc);
        pq_dist_cache<T>(h->dim, h->metric, (const T*)codebooks, m, n_bits, dcache.data());
        parallel_for(nq, nthreads, [&](size_t q) {
            const T* qv = (const T*)queries + q * h->dim;
            if (ties) ties[q] = 0;
            if (h->n == 0) {
                counts[q] = 0;
                return;
            }
            std::vector<float> lut(m * kc);
            float qn;
            pq_lookup(qv, h->dim, h->metric, (const T*)codebooks, m, n_bits, lut.data(), &qn);
            auto dist_fn = [&](size_t i) { return pq_adc(codes + i * enc, m, n_bits, h->metric, lut.data(), dcache.data(), qn); };
            size_t ep = h->greedy(0, dist_fn);
            ResultSet r = h->search_on_level(ep, 0, std::max(ef, k), dist_fn);
            const float qc = h->metric == ORC_L2SQR ? dot(qv, qv, h->dim) : vec_norm(qv, h->dim);
            ResultSet rs(k);
            for (const Pair& p : r.s) rs.add({h->d_cached(p.i, qv, qc), p.i});
            counts[q] = (uint32_t)emit(rs, k, ids + q * k, dists + q * k);
            if (ties) ties[q] = (uint32_t)(r.ties + rs.ties);   /* the walk's and pq_resort's */
        });
    });
    return 0;
}
int orc_hnsw_links0(const void* handle, int dtype, uint32_t* links0, uint32_t* len0) {
    D1(dtype, {
        const auto* h = (const Hnsw<T>*)handle;
        std::copy(h->level0.begin(), h->level0.end(), links0);
        for (size_t i = 0; i < h->n; ++i) len0[i] = (uint32_t)h->len[i][0];
    });
    return 0;
}
/* upper levels, per node levels 1..level in order: ulinks [sum(levels)][m], ulen [sum(levels)] */
int orc_hnsw_upper(const void* handle, int dtype, uint32_t* ulinks, uint32_t* ulen) {
    D1(dtype, {
        const auto* h = (const Hnsw<T>*)handle;
        size_t o = 0;
        for (size_t i = 0; i < h->n; ++i)
            for (size_t l = 1; l <= h->vec_level[i]; ++l) {
                std::copy(h->other[i].begin() + h->m * (l - 1), h->other[i].begin() + h->m * l, ulinks + o * h->m);
                ulen[o++] = (uint32_t)h->len[i][l];
            }
    });
    return 0;
}
void orc_hnsw_free(void* handle, int dtype) {
    D1(dtype, { delete (Hnsw<T>*)handle; });
}

/* candidate_pair.rs:127-140 */
float orc_recall(const uint64_t* gnd, size_t n_gnd, const uint64_t* pred, size_t n_pred) {
    std::set<uint64_t> p(pred, pred + n_pred);
    size_t hit = 0;
    for (size_t i = 0; i < n_gnd; ++i) hit += p.count(gnd[i]);
    return (float)hit / (float)n_gnd;
}

}  // extern "C"
