"""Every path-selection switch of tests/switch_matrix.py: same bits as the default path, and proof that the switch
changed the route.

Most switches are read once per process, so every (switch, value) runs its family's workload in a child process
(tests/switch_child.py) and is compared with the default child of that family:
  1. the kernel-launch fingerprint (name with template arguments, grid, block, shared memory) must differ, so the
     switch really selected other kernels or other launch shapes;
  2. every output must be bit-identical: ids, float32 distance bits, counts, PQ codes, HNSW links.
The default run of each family is itself checked against the CPU oracle, so "identical to the default" means correct.
"""
import ctypes as C
import os
import subprocess
import sys
from collections import Counter

import numpy as np
import pytest

from conftest import assert_knn_parity
from switch_matrix import SWITCHES, child_cases

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
CHILD = os.path.join(HERE, "switch_child.py")


def _child_env(extra):
    """The parent's environment without any VDB_* switch (VDB_LIB_PATH stays: it selects the build under test)."""
    env = {k: v for k, v in os.environ.items() if not k.startswith("VDB_") or k == "VDB_LIB_PATH"}
    env.update(extra)
    return env


def _run_child(family, out_dir, extra):
    tag = "-".join(f"{k}={v}" for k, v in extra.items()) or "default"
    out = os.path.join(str(out_dir), f"{family}-{tag}.npz")
    r = subprocess.run([sys.executable, CHILD, family, out], env=_child_env(extra), cwd=os.path.dirname(HERE),
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, f"child {family} {extra} exited {r.returncode}:\n{r.stdout[-4000:]}\n{r.stderr[-4000:]}"
    with np.load(out) as z:
        res = {k: z[k] for k in z.files}
    fp = Counter(res.pop("__fingerprint__").tolist())
    assert fp, "empty fingerprint"
    return res, fp


@pytest.fixture(scope="session")
def default_run(tmp_path_factory):
    cache = {}
    out_dir = tmp_path_factory.mktemp("switch_defaults")

    def get(family):
        if family not in cache:
            cache[family] = _run_child(family, out_dir, {})
        return cache[family]
    return get


@pytest.fixture(scope="module")
def child():
    sys.path.insert(0, HERE)
    import switch_child
    return switch_child


def _assert_same_bits(got, want, what):
    assert sorted(got) == sorted(want), f"{what}: output keys differ"
    for key in sorted(want):
        a, b = got[key], want[key]
        assert a.dtype == b.dtype and a.shape == b.shape, f"{what}: {key} is {a.dtype}{a.shape}, default {b.dtype}{b.shape}"
        if a.tobytes() != b.tobytes():
            rows = np.nonzero((a.reshape(len(a), -1).view(np.uint8) != b.reshape(len(b), -1).view(np.uint8)).any(1))[0] \
                if a.ndim else np.array([0])
            raise AssertionError(f"{what}: {key} differs from the default in {len(rows)} of {len(a) if a.ndim else 1} rows "
                                 f"(first {rows[:5].tolist()}): {a[rows[:2]] if a.ndim else a} vs {b[rows[:2]] if b.ndim else b}")


def _fp_diff(fp, ref):
    only = sorted((fp - ref).items())[:6]
    gone = sorted((ref - fp).items())[:6]
    return f"launched only with the switch: {only}; only by default: {gone}"


# ---- the default run of every family against the CPU oracle --------------------------------------------------------
def _check_flat(res, child, oracle):
    sets = child.flat_inputs()
    for s, metric, nq, k, redo in child.FLAT_CALLS:
        base, q = sets[s]
        key = child.flat_key(s, metric, nq, k, redo)
        got = (res[key + "/ids"], res[key + "/dist"], res[key + "/counts"])
        sel = np.r_[0:12, nq - 4:nq]
        want = oracle.flat_knn(base, q[sel], k, metric, nthreads=os.cpu_count() or 8)
        assert_knn_parity(base, q[sel], metric, tuple(a[sel] for a in got), want, oracle)
        assert (got[2] == min(k, len(base))).all(), key
    # the chunked 5000-query batches: the forced re-scan of every third query returns the same bits
    a, b = (child.flat_key("f32", "l2sqr", 5000, 10, r) for r in (0, 3))
    for part in ("ids", "dist", "counts"):
        assert res[a + "/" + part].tobytes() == res[b + "/" + part].tobytes()


def _check_merge(res, child, oracle):
    for i, (nlists, nq, k) in enumerate(child.MERGE_SHAPES):
        lists = child.merge_lists(nlists, nq, k, 8 + i)
        want = np.sort(lists.transpose(1, 0, 2).reshape(nq, -1), axis=1)[:, :k]
        key = f"merge/{nlists}x{nq}x{k}"
        assert (res[key + "/keys"] == want).all(), key
        valid = want != child.KEY_NONE
        assert (res[key + "/counts"] == valid.sum(1)).all(), key
        assert (res[key + "/ids"][valid] == (want[valid] & np.uint64(0xFFFFFFFF))).all(), key
        assert (res[key + "/ids"][~valid] == child.KEY_NONE).all(), key
    base, q = child.merge_sharded_inputs()
    for metric, nq, k in child.MERGE_SHARDED_CALLS:
        key = f"sharded/{metric}/nq{nq}/k{k}"
        sel = np.r_[0:min(nq, 16)]
        want = oracle.flat_knn(base, q[sel], k, metric, nthreads=os.cpu_count() or 8)
        got = (res[key + "/ids"], res[key + "/dist"], res[key + "/counts"])
        assert_knn_parity(base, q[sel], metric, tuple(a[sel] for a in got), want, oracle)


def _check_ivf(res, child, oracle):
    base, cent, q = child.ivf_inputs()
    for metric in dict.fromkeys(c[0] for c in child.IVF_CALLS):
        a = oracle.kmeans_assign(base, cent, metric, nthreads=os.cpu_count() or 8)
        assert (res[f"ivf/{metric}/assignment"] == a).all()
        off, mem = oracle.ivf_lists(a, child.IVF_NLIST)
        assert (np.diff(off)[:3] > 0).all()
        for m2, nq, k, nprobe in child.IVF_CALLS:
            if m2 != metric:
                continue
            key = f"ivf/{metric}/nq{nq}/k{k}/p{nprobe}"
            want = oracle.ivf_knn(base, cent, off, mem, q[:nq], k, nprobe, metric, nthreads=os.cpu_count() or 8)
            assert_knn_parity(base, q[:nq], metric, (res[key + "/ids"], res[key + "/dist"], res[key + "/counts"]), want, oracle)


def _check_pq(res, child, oracle):
    import lab_1806_vec_db_b200 as V
    sets = child.pq_inputs()
    for name, dtype, metric, m, n_bits in child.PQ_TABLES:
        base, q = sets[np.dtype(dtype).name]
        books = child.pq_books(V, base, m, n_bits)
        codes = oracle.pq_encode(base, books, m, n_bits, metric, nthreads=os.cpu_count() or 8)
        assert (res[f"pq/{name}/codes"] == codes).all(), name
        for nq, k, ef in child.PQ_CALLS:
            key = f"pq/{name}/nq{nq}/k{k}/ef{ef}"
            want = oracle.flat_knn_pq(base, codes, books, m, n_bits, q[:nq], k, ef, metric, nthreads=os.cpu_count() or 8)
            assert_knn_parity(base, q[:nq], metric, (res[key + "/ids"], res[key + "/dist"], res[key + "/counts"]), want, oracle)


def _check_hnsw(res, child, oracle):
    from oracle.oracle_py import HnswOracle
    base, q, levels = child.hnsw_inputs()
    assert (res["hnsw/levels"] == levels).all()
    ep, el = (int(x) for x in res["hnsw/enter_point"])
    cpu = HnswOracle.from_graph(base, "l2sqr", child.HNSW_M, child.HNSW_EFC, levels, res["hnsw/links0"], res["hnsw/len0"],
                                res["hnsw/ulinks"], res["hnsw/ulen"], ep, el)
    for ef in child.HNSW_EFS:
        ids, dd = res[f"hnsw/ef{ef}/ids"], res[f"hnsw/ef{ef}/dist"]
        oi, od, _ = cpu.knn(q, 10, ef, nthreads=os.cpu_count() or 8)
        same = ids.astype(np.int64) == oi.astype(np.int64)
        assert same.mean() >= 0.98, (ef, float(same.mean()))
        assert np.allclose(dd, od, rtol=1e-4, atol=1e-5)


CHECKS = {"flat": _check_flat, "merge": _check_merge, "ivf": _check_ivf, "pq": _check_pq, "hnsw": _check_hnsw}


@pytest.mark.parametrize("family", list(CHECKS))
def test_default_route_matches_the_oracle(family, default_run, child, oracle):
    res, _ = default_run(family)
    CHECKS[family](res, child, oracle)


# ---- every (switch, value): another route, the same bits -----------------------------------------------------------
@pytest.mark.parametrize("switch,value", child_cases(), ids=[f"{s}={v}" for s, v in child_cases()])
def test_switch_takes_another_route_with_the_same_bits(switch, value, default_run, tmp_path):
    family = SWITCHES[switch]["family"]
    want, fp0 = default_run(family)
    got, fp = _run_child(family, tmp_path, {switch: value})
    assert fp != fp0, f"{switch}={value} launched exactly the default kernels: the switch did not change the route"
    _assert_same_bits(got, want, f"{switch}={value} ({_fp_diff(fp, fp0)})")


# ---- VDB_GEMM_PART_RATIO: read per call ----------------------------------------------------------------------------
def test_row_part_ratio_changes_the_parts_not_a_bit(child, monkeypatch):
    """The filter pass cut into 3 row parts of shrinking size (ratio 0.5 and 0.2 of the previous part) returns the exact
    scan's bits, and the parts really differ from equal thirds (other contraction grids)."""
    import lab_1806_vec_db_b200 as V
    from lab_1806_vec_db_b200 import _lib as L
    base, q = child.flat_inputs()["f32"]
    q = q[:400]
    idx = V.FlatIndex.from_vec_set(base, "l2sqr")
    lib = L.lib()
    runs = {}
    try:
        L.check(lib.vdb_flat_set_path(1))
        scan = idx.knn_batch(q, 50)
        L.check(lib.vdb_flat_set_path(2))
        monkeypatch.setenv("VDB_GEMM_PARTS", "3")
        for ratio in (None, "0.5", "0.2"):
            if ratio is None:
                monkeypatch.delenv("VDB_GEMM_PART_RATIO", raising=False)
            else:
                monkeypatch.setenv("VDB_GEMM_PART_RATIO", ratio)
            runs[ratio] = child.fingerprint(lambda: idx.knn_batch(q, 50))
    finally:
        L.check(lib.vdb_flat_set_path(0))
    for ratio, (res, fp) in runs.items():
        for a, b in zip(res, scan):
            assert a.tobytes() == b.tobytes(), ratio
        if ratio is not None:
            assert fp != runs[None][1], f"VDB_GEMM_PART_RATIO={ratio} launched the kernels of equal parts"
