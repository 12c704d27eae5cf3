"""The IVF knn_pq reference (ivf_pq_reference.py) against its definition in terms of the Flat knn_pq oracle.

IVF knn_pq = FlatIndex::knn_pq (flat_index.rs:84-104) restricted to the rows of the n_probes nearest lists
(find_n_nearest, k_means.rs:174-191). So with every list probed it IS the Flat result, and with one list probed it is
the Flat result on that list's rows alone (ids mapped back: members are ascending, so the (value, id) order is kept)."""
import os

import numpy as np
import pytest

from ivf_pq_reference import ivf_knn_pq

NT = os.cpu_count() or 1
SHAPES = [("pq240", 240, 4, 960), ("pq7", 7, 4, 13), ("pq5b8", 5, 8, 13)]


def _setup(fixtures, golden, oracle, tag, m, n_bits, dimclip, metric):
    base = np.ascontiguousarray(fixtures["base"][:, :dimclip])
    queries = np.ascontiguousarray(fixtures["test"][:8, :dimclip])
    books = golden[f"{tag}_codebooks"]
    codes = oracle.pq_encode(base, books, m, n_bits, metric, nthreads=NT)
    cent = np.ascontiguousarray(base[7:23])
    off, mem = oracle.ivf_lists(oracle.kmeans_assign(base, cent, metric, nthreads=NT), 16)
    return base, queries, books, codes, cent, off, mem


@pytest.mark.parametrize("tag,m,n_bits,dimclip", SHAPES)
@pytest.mark.parametrize("metric", ["l2sqr", "cosine"])
def test_all_lists_probed_is_flat_knn_pq(fixtures, golden, oracle, tag, m, n_bits, dimclip, metric):
    base, queries, books, codes, cent, off, mem = _setup(fixtures, golden, oracle, tag, m, n_bits, dimclip, metric)
    for k, ef in ((10, 40), (10, 4), (3, 2000)):
        want = oracle.flat_knn_pq(base, codes, books, m, n_bits, queries, k, ef, metric, nthreads=NT)
        for n_probes in (16, 50):
            got, _ = ivf_knn_pq(oracle, base, codes, books, m, n_bits, cent, off, mem, queries, k, ef, n_probes, metric)
            assert (got[0] == want[0]).all() and (got[2] == want[2]).all()
            assert (got[1].view(np.uint32) == want[1].view(np.uint32)).all()


@pytest.mark.parametrize("tag,m,n_bits,dimclip", SHAPES)
@pytest.mark.parametrize("metric", ["l2sqr", "cosine"])
def test_one_list_probed_is_flat_knn_pq_on_its_rows(fixtures, golden, oracle, tag, m, n_bits, dimclip, metric):
    base, queries, books, codes, cent, off, mem = _setup(fixtures, golden, oracle, tag, m, n_bits, dimclip, metric)
    k, ef = 10, 40
    (got_i, got_d, got_c), _ = ivf_knn_pq(oracle, base, codes, books, m, n_bits, cent, off, mem, queries, k, ef, 1, metric)
    for q in range(queries.shape[0]):
        c = int(oracle.find_n_nearest(queries[q], cent, 1, metric)[0])
        rows = mem[int(off[c]):int(off[c + 1])].astype(np.int64)
        wi, wd, wc = oracle.flat_knn_pq(base[rows], codes[rows], books, m, n_bits, queries[q:q + 1], k, ef, metric)
        n = int(wc[0])
        assert int(got_c[q]) == n == min(k, rows.size)
        assert (got_i[q, :n].astype(np.int64) == rows[wi[0, :n].astype(np.int64)]).all()
        assert (got_d[q, :n].view(np.uint32) == wd[0, :n].view(np.uint32)).all()
