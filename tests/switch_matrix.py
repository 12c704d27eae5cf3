"""Every VDB_* environment switch the CUDA sources read, and how the suite proves it changes no result.

Plain data, importable without a GPU. `SWITCHES` are the path-selection switches whose alternative routes are run by
tests/test_switches_gpu.py: each (switch, value) runs its family's workload (tests/switch_child.py) in a child process
and must launch a different set of kernels than the default run while returning the same bits. `OTHER` lists the
remaining switches and where they are covered or why they need no parity case. tests/test_switches_cpu.py fails when a
`getenv("VDB_...")` in lab_1806_vec_db_b200/csrc is in neither table.

read: "process" = read once per process (a `static const` in the source: only a fresh process sees a new value);
      "call"    = read on every call (tests may set it with monkeypatch inside one process).
"""

SWITCHES = {
    # ---- Flat tensor path (flat_gemm.cu) ----
    "VDB_GEMM_CTAS": dict(values=("1",), family="flat", read="process",
                          route="single-CTA contraction for batches of > 128 queries (default: CTA pairs)"),
    "VDB_GEMM_SMALL_PAIRS": dict(values=("1",), family="flat", read="process",
                                 route="CTA pairs for batches of 3-128 queries (default: single CTAs)"),
    "VDB_GEMM_TPS": dict(values=("1", "8"), family="flat", read="process",
                         route="row tiles per slab of the filter pass (default 4, capped by plan_gemm)"),
    "VDB_GEMM_CHUNKS": dict(values=("2", "3"), family="flat", read="process",
                            route="query chunks pipelined over two worker streams (batches of >= 4096 queries), "
                                  "then the exact re-scan of flagged queries"),
    "VDB_GEMM_SAMPLE_N": dict(values=("4096",), family="flat", read="process",
                              route="a smaller threshold sample (default max(2048, n / 30) rows, at most 32768)"),
    "VDB_GEMM_SAMPLE_SUBN": dict(values=("256",), family="flat", read="process",
                                 route="sub-sample size of the two-level sample selection (k large: j > 16)"),
    "VDB_GEMM_SAMPLE_TPS": dict(values=("1", "32"), family="flat", read="process",
                                route="row tiles per slab of the one-launch sample pass (j <= 16)"),
    "VDB_GEMM_PART_RATIO": dict(values=("0.5", "0.2"), family="flat", read="call",
                                route="share of slabs per row part under VDB_GEMM_PARTS=3 (tested in-process)"),
    # ---- key merges (flat_scan.cu; multi.cu and the sharded thresholds call them) ----
    "VDB_MERGE_GENERIC": dict(values=("1",), family="merge", read="process",
                              route="the generic sort-based key merge instead of the rank merge of sorted lists"),
    # ---- IVF probe scan (flat_gemm.cu, ivf.cu) ----
    "VDB_IVF_CTAS": dict(values=("0", "2"), family="ivf", read="process",
                         route="query tiles of the tensor probe scan on CTA pairs (0: > 128 queries, 2: all)"),
    "VDB_IVF_SUBSET": dict(values=("1",), family="ivf", read="process",
                           route="thresholds from an exact subset scan where the list sample is the default"),
    "VDB_IVF_NO_TENSOR": dict(values=("1",), family="ivf", read="process",
                              route="FP32 list-major scan instead of the tensor probe scan"),
    # ---- PQ (pq.cu, pq_gemm.cu) ----
    "VDB_ADC_OLD": dict(values=("1",), family="pq", read="process",
                        route="per-CTA top-k ADC scan for batches on large shards (default: global threshold)"),
    "VDB_ADC_NQ": dict(values=("1", "2"), family="pq", read="process",
                       route="queries per CTA of the per-CTA ADC scan (default 4)"),
    "VDB_PQ_SELECT_OLD": dict(values=("1",), family="pq", read="process",
                              route="sort-based threshold selection of the global-threshold scan"),
    "VDB_PQ_NO_TENSOR": dict(values=("1",), family="pq", read="process",
                             route="FP32 global-threshold scan instead of the tensor-core filter"),
    "VDB_PQ_TENSOR_MIN_NQ": dict(values=("4", "100000"), family="pq", read="process",
                                 route="smallest batch of the tensor-core filter (default 32)"),
    "VDB_PQ_CTAS": dict(values=("2",), family="pq", read="process",
                        route="CTA-pair variant of the one-hot PQ contraction"),
    "VDB_PQ_GEN": dict(values=("1", "2"), family="pq", read="process",
                       route="1- and 2-warpgroup generators of the one-hot PQ contraction (default 4)"),
    "VDB_PQ_ENCODE_OLD": dict(values=("1",), family="pq", read="process",
                              route="generic PQ encoder on 4-bit tables of <= 8-dim sub-vectors"),
    # ---- HNSW (hnsw.cu) ----
    "VDB_HNSW_SMALL_HASH_EF": dict(values=("0", "200"), family="hnsw", read="process",
                                   route="largest ef of the 8192-slot visited set (default 448); only values that "
                                         "move a search to a LARGER set are tested"),
}

# Switches without a child-process parity case here, and why.
OTHER = {
    "VDB_GEMM_KIND": ("call", "tests/test_gemm_gpu.py::test_tensor_path_identical_to_exact_scan"),
    "VDB_GEMM_PARTS": ("call", "tests/test_gemm_gpu.py::test_round2_stages_do_not_change_a_bit"),
    "VDB_GEMM_PRUNE": ("call", "tests/test_gemm_gpu.py::test_round2_stages_do_not_change_a_bit"),
    "VDB_GEMM_RARE_PER_SCORE": ("call", "tests/test_gemm_gpu.py::test_round2_stages_do_not_change_a_bit"),
    "VDB_GEMM_SAMPLE_2L": ("call", "tests/test_gemm_gpu.py::test_round2_stages_do_not_change_a_bit"),
    "VDB_SCAN_FUSE": ("call", "tests/test_flat_gpu.py::test_fused_scan_tail_equals_the_separate_merge"),
    "VDB_PQ_NO_DECODE": ("call", "tests/test_index_gpu.py::test_pq_decoded_contraction_large_shard"),
    "VDB_MG_GLOBAL_PRUNE": ("call", "tests/test_multi_gpu.py::test_global_pruning_bound_changes_no_bit_and_gathers_fewer_rows"),
    "VDB_HNSW_HASH_SLOTS": ("process", "test hook: forces the first visited-set size of every search; "
                                       "tests/test_hnsw_gpu.py::test_a_full_visited_set_is_searched_again_not_a_silent_loss"),
    "VDB_MG_TRACE": ("process", "diagnostic print of the sharded search's host phase times; selects no kernel"),
}

FAMILIES = ("flat", "merge", "ivf", "pq", "hnsw")


def child_cases():
    """(switch, value) pairs that run in a child process."""
    return [(name, v) for name, s in SWITCHES.items() if s["read"] == "process" for v in s["values"]]
