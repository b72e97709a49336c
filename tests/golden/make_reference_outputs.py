"""Stores what the UNMODIFIED reference CPU library (oracle/_ref, built by oracle/Makefile) answers for the
inputs of the tests that compare with it, so that those tests run where the library is absent:

    python tests/golden/make_reference_outputs.py cpu
        -> tests/golden/reference_outputs.npz            (test_abi.py, test_oracle.py; no GPU needed)
    python tests/golden/make_reference_outputs.py fullsize OUT.npz
        -> the BASELINE-size configs of test_fullsize_gpu.py (needs a B200: the inputs and the GPU index
           contents that the reference is handed are made on the device; copy OUT.npz to
           tests/golden/reference_outputs_fullsize.npz)

The inputs are not stored: the tests regenerate them from the same seeds with the helpers imported below.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref  # noqa: E402


def _store_ivfpq(out, prefix, ivf, nlist, xb):
    """the reference's IndexIVFPQ content: centroids, PQ codebooks, the list of every vector (ids are 0..n-1 in insertion
    order, so every list holds its ids ascending) and the codes -- as the oracle's encoding of each residual plus the
    rows where the reference's code differs (fp near-ties), which rebuilds the reference's lists byte for byte"""
    from oracle import oracle_np as o

    cent, pq = ivf.centroids(), ivf.pq_centroids()
    n, M = xb.shape[0], pq.shape[0]
    assign = np.full(n, -1, dtype=np.int64)
    codes = np.zeros((n, M), dtype=np.uint8)
    for l in range(nlist):
        c, ids = ivf.get_list(l)
        assert (np.diff(ids) > 0).all()
        assign[ids] = l
        codes[ids] = c.reshape(ids.size, M)
    assert (assign >= 0).all() and nlist <= 256
    rows = np.flatnonzero((o.pq_encode(xb - cent[assign], pq) != codes).any(axis=1))
    out[prefix + "_centroids"], out[prefix + "_pq"] = cent, pq
    out[prefix + "_list"] = assign.astype(np.uint8)
    out[prefix + "_patch_rows"], out[prefix + "_patch_codes"] = rows.astype(np.int32), codes[rows]


def _ids32(D, I):
    """ids fit in int32 in every stored result: half the bytes"""
    assert I.max() < 2**31
    return D, I.astype(np.int32)


def cpu():
    from tests.test_abi import merge_trials
    from tests.test_oracle import flat_live_inputs, precomputed_form_inputs, precomputed_onoff_inputs

    out = {}
    merged = [_ids32(*ref.merge_knn_results(allD, allI, metric)) for allD, allI, metric in merge_trials()]
    out["merge_D"] = np.concatenate([D.ravel() for D, _ in merged])  # trial after trial, each [n, k] row-major
    out["merge_I"] = np.concatenate([I.ravel() for _, I in merged])

    for i, (xb, xq, k, metric) in enumerate(flat_live_inputs()):
        idx = ref.IndexFlat(xb.shape[1], metric)
        idx.add(xb)
        out["flat_%d_D" % i], out["flat_%d_I" % i] = _ids32(*idx.search(xq, k))

    xb, xq = precomputed_onoff_inputs()
    ivf = ref.IndexIVFPQ(16, 8, 4, 8, 1)
    ivf.set_cp(niter=4)
    ivf.set_pq_cp(niter=4)
    ivf.train(xb)
    ivf.add(xb)
    ivf.set_nprobe(3)
    ivf.set_precomputed_table(1)
    out["onoff_D1"], out["onoff_I1"] = _ids32(*ivf.search(xq, 10))
    ivf.set_precomputed_table(0)
    out["onoff_D0"], out["onoff_I0"] = _ids32(*ivf.search(xq, 10))
    _store_ivfpq(out, "onoff", ivf, 8, xb)

    xb, xq = precomputed_form_inputs()
    ivf = ref.IndexIVFPQ(32, 16, 8, 8, 1)
    ivf.set_cp(niter=4)
    ivf.set_pq_cp(niter=4)
    ivf.train(xb)
    ivf.add(xb)
    ivf.set_nprobe(4)
    ivf.set_precomputed_table(1)
    out["pcform_D"], out["pcform_I"] = _ids32(*ivf.search(xq, 10))
    _store_ivfpq(out, "pcform", ivf, 16, xb)

    path = os.path.join(ROOT, "tests", "golden", "reference_outputs.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes;", ref.compile_options())


def _clone_search(cpu_index, gpu_index, nlist, xq, k, nprobe):
    """hand the GPU index's lists to the reference index and search it"""
    for l in range(nlist):
        ids = gpu_index.getListIndices(l)
        if ids.size:
            cpu_index.add_entries(l, ids, gpu_index.getListVectorData(l))
    assert cpu_index.ntotal == gpu_index.ntotal
    cpu_index.set_nprobe(nprobe)
    return _ids32(*cpu_index.search(xq, k))


def fullsize(path):
    import torch

    import faiss_b200 as fb
    from tests.test_fullsize_gpu import _sample_queries, flat_10m_inputs, ivfflat_10m_index, ivfpq_100m_index

    res = fb.StandardGpuResources()
    ref.set_omp_threads(16)
    out = {}
    k, d, nlist = 100, 128, 4096

    xb, xq, pick = flat_10m_inputs(torch)
    out["flat_D"], out["flat_I"] = _ids32(*ref.knn(xq[pick].cpu().numpy(), xb.cpu().numpy(), k, 1))
    xbi = torch.floor(xb * 16)
    del xb
    out["flatint_D"], out["flatint_I"] = _ids32(*ref.knn(torch.floor(xq[pick] * 16).cpu().numpy(), xbi.cpu().numpy(), k, 1))
    del xbi
    torch.cuda.empty_cache()
    print("flat done", flush=True)

    xq, pick = _sample_queries(torch, 10_000, d, 1235)
    xqs = xq[pick].cpu().numpy()
    idx = ivfflat_10m_index(torch, fb, res)
    cpu = ref.IndexIVFFlat(d, nlist, 1)
    cpu.set_centroids(idx.getCoarseCentroids())
    cpu.set_is_trained(True)
    out["ivfflat_D"], out["ivfflat_I"] = _clone_search(cpu, idx, nlist, xqs, k, 64)
    del idx, cpu
    torch.cuda.empty_cache()
    print("ivfflat done", flush=True)

    M = 32
    idx = ivfpq_100m_index(torch, fb, res)
    cpu = ref.IndexIVFPQ(d, nlist, M, 8, 1)
    cpu.set_centroids(idx.getCoarseCentroids())
    cpu.set_pq_centroids(idx.getPQCentroids())
    cpu.set_is_trained(True)
    cpu.set_precomputed_table(0)  # 0 = the reference's own rule
    out["ivfpq_D"], out["ivfpq_I"] = _clone_search(cpu, idx, nlist, xqs, k, 32)
    print("ivfpq done", flush=True)

    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes;", ref.compile_options())


if __name__ == "__main__":
    if sys.argv[1:2] == ["cpu"]:
        cpu()
    elif sys.argv[1:2] == ["fullsize"]:
        fullsize(sys.argv[2])
    else:
        sys.exit(__doc__)
