"""The C-ABI library loads and exports every symbol include/faiss_b200_c.h declares; host-side
logic of the path (no GPU compute calls here)."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    txt = open(os.path.join(ROOT, "include", "faiss_b200_c.h")).read()
    return sorted(s for s in set(re.findall(r"FB200_API\s+[^;(]*?\b(\w+)\s*\(", txt)) if s != "__attribute__")


def test_header_declares_functions():
    syms = _declared_symbols()
    assert len(syms) > 50
    for must in ("faiss_Index_search", "faiss_GpuIndexFlat_new", "faiss_GpuIndexIVFPQ_new",
                 "faiss_StandardGpuResources_new", "faiss_IndexShards_add_shard", "b200_topk_merge"):
        assert must in syms


def test_library_exports_every_declared_symbol():
    import faiss_b200 as fb

    missing = [s for s in _declared_symbols() if not hasattr(fb.lib, s)]
    assert not missing, "declared but not exported: %s" % missing
    assert b"sm_100a" in fb.lib.faiss_b200_version()


def test_error_convention_without_gpu():
    """null handles -> FAISS_EXCEPT (-2) + message, as c_api/macros_impl.h:22-36"""
    import faiss_b200 as fb

    rc = fb.lib.faiss_Index_search(None, ctypes.c_int64(1), None, ctypes.c_int64(1), None, None)
    assert rc == -2
    assert b"null index handle" in fb.lib.faiss_get_last_error()


def test_product_does_not_import_oracle():
    """the product path must never route through oracle/"""
    for root, _, files in os.walk(os.path.join(ROOT, "faiss_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                txt = open(os.path.join(root, f), errors="ignore").read()
                assert "oracle_np" not in txt and "libfaiss_ref" not in txt and "import oracle" not in txt, f


def test_host_rand_perm_matches_reference(golden):
    import faiss_b200 as fb

    perm = np.empty(1000, dtype=np.int32)
    assert fb.lib.faiss_b200_rand_perm(perm.ctypes.data_as(ctypes.POINTER(ctypes.c_int)), ctypes.c_size_t(1000), ctypes.c_int64(42)) == 0
    assert np.array_equal(perm, golden["rand_perm_1000_s42"])


def test_host_merge_matches_reference(golden):
    from faiss_b200.distributed import merge_host

    D, I = merge_host(golden["merge_allD"], golden["merge_allI"], 5, 1)
    assert np.array_equal(I, golden["merge_I"])
    assert np.array_equal(D, golden["merge_D"])


def test_host_split_clusters_matches_oracle():
    import faiss_b200 as fb
    from oracle import oracle_np as o

    rs = np.random.RandomState(3)
    k, d, n = 12, 6, 500
    h = rs.randint(1, 60, size=k).astype(np.float32)
    h[[2, 7, 8]] = 0
    c = rs.rand(k, d).astype(np.float32)
    h2, c2 = h.copy(), c.copy()
    ns = ctypes.c_int()
    fp = ctypes.POINTER(ctypes.c_float)
    assert fb.lib.faiss_b200_split_clusters(ctypes.c_size_t(d), ctypes.c_size_t(k), ctypes.c_size_t(n), h.ctypes.data_as(fp), c.ctypes.data_as(fp), ctypes.byref(ns)) == 0
    ns2 = o.split_clusters(d, k, n, h2, c2)
    assert ns.value == ns2 == 3
    assert np.array_equal(h, h2)
    assert np.allclose(c, c2, rtol=1e-6)


def test_shard_bounds_contiguous():
    from faiss_b200.distributed import shard_bounds

    n, w = 1003, 8
    b = [shard_bounds(n, r, w) for r in range(w)]
    assert b[0][0] == 0 and b[-1][1] == n
    assert all(b[i][1] == b[i + 1][0] for i in range(w - 1))


def test_cloner_shard_ivf_lists_rules():
    """shard_type 1 / 2 / 4 of ToGpuClonerMultiple::copy_ivf_shard (faiss/gpu/GpuCloner.cpp:287-322) on the
    ArrayInvertedLists payload: a partition, list order kept, the reference's boundaries"""
    from faiss_b200 import cloner

    rs = np.random.RandomState(2)
    nlist, code_size, ntotal = 13, 6, 1000
    assign = rs.randint(0, nlist, ntotal)
    all_ids = rs.permutation(ntotal).astype(np.int64)
    ids = [all_ids[assign == l] for l in range(nlist)]
    codes = [rs.randint(0, 256, (a.size, code_size)).astype(np.uint8).reshape(-1) for a in ids]
    for st in (cloner.SHARD_BY_ID_MOD, cloner.SHARD_BY_ID_RANGE, cloner.SHARD_BY_LIST_RANGE):
        for n in (1, 2, 3, 8):
            parts = cloner.shard_ivf_lists(codes, ids, code_size, n, st)
            assert len(parts) == n
            for l in range(nlist):
                got_ids = np.concatenate([p[1][l] for p in parts])
                assert sorted(got_ids.tolist()) == sorted(ids[l].tolist())  # partition of the list
                for i, (ci, ii) in enumerate(parts):
                    # order inside the list is the original order, codes travel with their ids
                    pos = {int(v): j for j, v in enumerate(ids[l])}
                    js = [pos[int(v)] for v in ii[l]]
                    assert js == sorted(js)
                    ref_codes = codes[l].reshape(-1, code_size)[js].reshape(-1)
                    assert np.array_equal(ci[l], ref_codes)
                    if st == cloner.SHARD_BY_ID_MOD:
                        assert ((ii[l] % n) == i).all()
                    elif st == cloner.SHARD_BY_ID_RANGE:
                        assert ((ii[l] >= i * ntotal // n) & (ii[l] < (i + 1) * ntotal // n)).all()
                    else:
                        assert ii[l].size == (ids[l].size if i * nlist // n <= l < (i + 1) * nlist // n else 0)
    with pytest.raises(ValueError):
        cloner.shard_ivf_lists(codes, ids, code_size, 2, 3)


def merge_trials():
    """60 random sets of shard results with heavy distance ties, -1 padding (shards with fewer than k results) and both
    metrics: (allD [ns, n, k], allI, metric).  tests/golden/make_reference_outputs.py stores the reference's merge of each."""
    rs = np.random.RandomState(123)
    for trial in range(60):
        ns, n, k = rs.randint(1, 6), rs.randint(1, 9), rs.randint(1, 17)
        metric = int(rs.randint(0, 2))
        allD = np.empty((ns, n, k), dtype=np.float32)
        allI = np.empty((ns, n, k), dtype=np.int64)
        for s in range(ns):
            for q in range(n):
                m = rs.randint(0, k + 1)  # valid results of this shard for this query
                d = np.sort(rs.randint(0, 6, m).astype(np.float32))  # few distinct values: many ties
                if metric == 0:
                    d = d[::-1]
                ids = rs.permutation(1000)[:m].astype(np.int64) + 1000 * s  # ids disjoint across shards
                pad_d = np.float32(np.finfo(np.float32).max) if metric == 1 else np.float32(-np.finfo(np.float32).max)
                allD[s, q] = np.concatenate([d, np.full(k - m, pad_d, dtype=np.float32)])
                allI[s, q] = np.concatenate([ids, np.full(k - m, -1, dtype=np.int64)])
        yield allD, allI, metric


def test_host_merge_property_vs_reference_live(ref_outputs):
    """merge_knn_results (faiss/utils/Heap.cpp:166-238, results stored from the reference library) vs the library's
    host merge on merge_trials().
    Distances must be identical; ids identical wherever the distance is not tied (the reference's heap
    merge leaves the order inside a run of equal distances unspecified; ours is (distance, id))."""
    from faiss_b200.distributed import merge_host

    o0 = 0
    for allD, allI, metric in merge_trials():
        n, k = allD.shape[1], allD.shape[2]
        rD = ref_outputs["merge_D"][o0 : o0 + n * k].reshape(n, k)
        rI = ref_outputs["merge_I"][o0 : o0 + n * k].reshape(n, k)
        o0 += n * k
        D, I = merge_host(allD, allI, k, metric)
        valid = rI >= 0
        assert np.array_equal(valid, I >= 0)
        assert np.array_equal(D[valid], rD[valid])
        for q in range(n):
            for v in np.unique(D[q][valid[q]]):
                sel = (D[q] == v) & valid[q]
                # same multiset of ids per tied run unless the run is cut by the k boundary
                if sel[-1] and valid[q][-1]:
                    continue
                assert sorted(I[q][sel].tolist()) == sorted(rI[q][sel].tolist())
    assert o0 == ref_outputs["merge_D"].size
