"""IVF knn_pq reference, composed from the CPU oracle's reference functions (test infrastructure).

The reference has no IVF knn_pq; the library defines it (INTEGRATION.md) as FlatIndex::knn_pq (flat_index.rs:84-104)
restricted to the rows of the n_probes nearest lists (find_n_nearest, k_means.rs:174-191):
  1. find_n_nearest;
  2. the union of the probed lists' members, ascending (the visiting order is the tie rule of ResultSet::add);
  3. the max(ef, k) best (ADC, id) over those rows (oracle.flat_adc_topk on the rows' codes: ADC in the reference
     arithmetic, pq_table.rs:239-301);
  4. pq_resort (candidate_pair.rs:102-108): exact distances in candidate order into a bounded ResultSet of k.
Every float is computed by the oracle library (-ffp-contract=off); this module only selects and orders.
"""
import numpy as np


def _result_set_add(rs, k, d, i):
    """ResultSet::add (candidate_pair.rs:61-74): rs is kept sorted by (distance, id); a full set takes a pair only when
    its distance is strictly below the last one's (NaN orders last)."""
    key = (bool(np.isnan(d)), 0.0 if np.isnan(d) else float(d), i, d)
    if len(rs) < k:
        rs.append(key)
        rs.sort()
    elif rs and key[:2] < rs[-1][:2]:
        rs[-1] = key
        rs.sort()


def ivf_knn_pq(oracle, base, codes, codebooks, m, n_bits, centroids, offsets, members, queries, k, ef, n_probes, metric):
    """Returns ((ids [nq,k] u64, dist [nq,k] f32, counts [nq] u32), (cand_ids [nq,kk], cand_adc [nq,kk], cand_counts [nq]))
    with kk = max(ef, k); unused entries are UINT64_MAX / NaN as the oracle emits them."""
    assert n_probes > 0
    base, codes, queries = np.ascontiguousarray(base), np.ascontiguousarray(codes), np.ascontiguousarray(queries)
    offsets, members = np.asarray(offsets, np.int64), np.asarray(members, np.int64)
    nq, dim, kk = queries.shape[0], base.shape[1], max(ef, k)
    dc = oracle.pq_dist_cache(dim, codebooks, m, n_bits, metric)
    ids = np.full((nq, k), np.iinfo(np.uint64).max, np.uint64)
    dd = np.full((nq, k), np.nan, np.float32)
    cnt = np.zeros(nq, np.uint32)
    cids = np.full((nq, kk), np.iinfo(np.uint64).max, np.uint64)
    cdd = np.full((nq, kk), np.nan, np.float32)
    ccnt = np.zeros(nq, np.uint32)
    for q in range(nq):
        probes = oracle.find_n_nearest(queries[q], centroids, n_probes, metric)
        rows = np.sort(np.concatenate([members[offsets[c]:offsets[c + 1]] for c in probes.astype(np.int64)]))
        lut, qc = oracle.pq_lookup(queries[q], codebooks, m, n_bits, metric)
        if rows.size:
            local, adc = oracle.flat_adc_topk(codes[rows], m, n_bits, metric, lut, dc, qc, kk)
            cand = rows[local.astype(np.int64)]
        else:
            cand, adc = np.zeros(0, np.int64), np.zeros(0, np.float32)
        ccnt[q] = cand.size
        cids[q, :cand.size], cdd[q, :cand.size] = cand, adc
        rs = []
        for i in cand:
            _result_set_add(rs, k, np.float32(oracle.distance(queries[q], base[i], metric)), int(i))
        cnt[q] = len(rs)
        for j, (_, _, i, d) in enumerate(rs):
            ids[q, j], dd[q, j] = i, d
    return (ids, dd, cnt), (cids, cdd, ccnt)
