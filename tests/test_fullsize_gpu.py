"""Full-size (BASELINE.json configs) property tests on a B200, through the C ABI.

The oracle cannot answer 10M x 10k in test time, so these use size-independent properties of the path:
equality of the tcgen05 path with the exact fp32 kernel (bit for bit) on a query sample, self-queries,
sortedness / uniqueness, shard-and-merge == unsharded, search == search_preassigned
(faiss/gpu/test/test_gpu_index.py:190-194), batch-size invariance and run-to-run determinism.
Synthetic data, generated on the device in seeded chunks."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _rows(torch, n, d, seed0, chunk=1_000_000):
    out = torch.empty((n, d), dtype=torch.float32, device="cuda")
    for c0 in range(0, n, chunk):
        g = torch.Generator(device="cuda")
        g.manual_seed(seed0 + c0 // chunk)
        c1 = min(n, c0 + chunk)
        out[c0:c1] = torch.rand((c1 - c0, d), dtype=torch.float32, device="cuda", generator=g)
    return out


def test_flat_l2_10m_properties(res):
    """configs[1]: GpuIndexFlatL2, N=10M, d=128, nq=10k, k=100"""
    import torch

    import faiss_b200 as fb

    N, d, nq, k = 10_000_000, 128, 10_000, 100
    xb = _rows(torch, N, d, 1234)
    g = torch.Generator(device="cuda")
    g.manual_seed(77)
    xq = torch.rand((nq, d), dtype=torch.float32, device="cuda", generator=g)
    # 64 self-queries: a database row must come back first, at distance exactly 0
    self_rows = torch.arange(0, N, N // 64, device="cuda")[:64]
    xq[:64] = xb[self_rows]
    idx = fb.GpuIndexFlatL2(res, d)
    idx.add(xb)
    D, I = idx.search(xq, k)
    info = idx.lastSearchInfo()
    assert info["tensor_cores"] == 1
    assert info["fallback_queries"] <= nq // 100
    # sorted, in range, no duplicate ids per query
    assert bool((D[:, 1:] >= D[:, :-1]).all())
    assert bool(((I >= 0) & (I < N)).all())
    srt = torch.sort(I, dim=1).values
    assert bool((srt[:, 1:] != srt[:, :-1]).all())
    assert torch.equal(I[:64, 0], self_rows) and bool((D[:64, 0] == 0).all())
    # run-to-run determinism
    D2, I2 = idx.search(xq, k)
    assert torch.equal(D, D2) and torch.equal(I, I2)
    # the tcgen05 path == the exact fp32 kernel, bit for bit, on a query sample
    sample = torch.cat([torch.arange(0, 128, device="cuda"), torch.arange(nq - 128, nq, device="cuda")])
    idx.setUseTensorCores(False)
    De, Ie = idx.search(xq[sample], k)
    assert idx.lastSearchInfo()["tensor_cores"] == 0
    assert torch.equal(I[sample], Ie) and torch.equal(D[sample], De)
    idx.setUseTensorCores(True)
    # batch-size invariance of the tcgen05 path (different round schedule, same answer)
    Db, Ib = idx.search(xq[:1000], k)
    assert torch.equal(Db, D[:1000]) and torch.equal(Ib, I[:1000])
    # shard + merge == unsharded (IndexShards semantics, faiss/gpu/test/test_multi_gpu.py:23-43)
    del idx
    half = N // 2
    parts = []
    for r0, r1 in ((0, half), (half, N)):
        sh = fb.GpuIndexFlatL2(res, d)
        sh.add(xb[r0:r1])
        parts.append(sh.search(xq[:2000], k))
        del sh
    allD = torch.stack([p[0] for p in parts], dim=1).contiguous()  # [nq, nshard, k]
    allI = torch.stack([p[1] for p in parts], dim=1).contiguous()
    offs = torch.tensor([0, half], dtype=torch.int64, device="cuda")
    mD, mI = fb.topk_merge(res, allD, allI, k, fb.METRIC_L2, id_offsets=offs)
    assert torch.equal(mD, D[:2000]) and torch.equal(mI, I[:2000])


def test_ivfpq_100m_properties(res):
    """configs[3]: GpuIndexIVFPQ, N=100M, d=128, nlist=4096, M=32, nprobe=32 (train 1M, add 100M)"""
    import torch

    import faiss_b200 as fb

    N, d, nlist, M, nprobe, nq, k = 100_000_000, 128, 4096, 32, 32, 4000, 100
    idx = fb.GpuIndexIVFPQ(res, d, nlist, M, 8, fb.METRIC_L2)
    idx.setClustering(niter=6)
    idx.setPQClustering(niter=6)
    xt = _rows(torch, 1 << 19, d, 4321)
    idx.train(xt)
    del xt
    idx.reserveMemory(N + N // 8)
    CH = 2_000_000
    probe_rows = None
    for c0 in range(0, N, CH):
        xb = _rows(torch, min(CH, N - c0), d, 1234 + c0 // CH)
        if c0 == 0:
            probe_rows = xb[:32].clone()
        idx.add(xb)
        del xb
    assert idx.ntotal == N
    lens = np.array([idx.getListLength(l) for l in range(0, nlist, 64)])
    assert lens.min() > 0
    g = torch.Generator(device="cuda")
    g.manual_seed(99)
    xq = torch.rand((nq, d), dtype=torch.float32, device="cuda", generator=g)
    xq[:32] = probe_rows  # stored vectors as queries
    idx.nprobe = nprobe
    D, I = idx.search(xq, k)
    assert bool((D[:, 1:] >= D[:, :-1]).all())
    assert bool(((I >= 0) & (I < N)).all())
    # a stored vector finds itself (ids are insertion order) within its top results: its own code is the
    # nearest reproduction of it unless another vector shares the list and a closer code
    hit = (I[:32, :10] == torch.arange(32, device="cuda").unsqueeze(1)).any(dim=1)
    assert int(hit.sum()) >= 30
    # determinism + batch-size invariance (one CTA per query at nq=4000, probes split at nq=100)
    D2, I2 = idx.search(xq, k)
    assert torch.equal(D, D2) and torch.equal(I, I2)
    Db, Ib = idx.search(xq[:100], k)
    assert torch.equal(Db, D[:100])
    same = Ib == I[:100]
    tied = torch.zeros_like(same)
    tied[:, 1:] |= D[:100, 1:] == D[:100, :-1]
    tied[:, :-1] |= D[:100, :-1] == D[:100, 1:]
    assert bool((same | tied).all())
    # search == search_preassigned with the coarse quantiser's own assignment, bit-exact
    cent = torch.from_numpy(idx.getCoarseCentroids()).cuda()
    cd = torch.cdist(xq[:500], cent) ** 2
    cD, cI = cd.topk(nprobe, dim=1, largest=False)
    D3, I3 = idx.search_preassigned(xq[:500], k, cI.contiguous(), cD.contiguous())
    # torch's coarse assignment can differ from the index's on fp near-ties of the 32nd probe: the
    # queries whose probe sets agree must match bit for bit, and that must be the large majority
    Dq, Iq = idx.search(xq[:500], k)
    eq = (D3 == Dq).all(dim=1) & (I3 == Iq).all(dim=1)
    assert float(eq.float().mean()) > 0.9


# ------------------------------------------------------------------------------------------------
# BASELINE-size configs against the reference itself on sampled queries: the answers of the reference CPU library
# (oracle/_ref) for exactly these inputs and index contents are stored in tests/golden/reference_outputs_fullsize.npz
# by tests/golden/make_reference_outputs.py, which builds them with the helpers below.
# Model: faiss/gpu/test/TestUtils.cpp:158-226 (compareLists), TestGpuIndexFlat.cpp, TestGpuIndexIVFFlat.cpp,
# TestGpuIndexIVFPQ.cpp -- the GPU index and the CPU index hold the SAME data; 64 sampled queries.
# ------------------------------------------------------------------------------------------------
def _sample_queries(torch, nq, d, seed, n=64):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    xq = torch.rand((nq, d), dtype=torch.float32, device="cuda", generator=g)
    pick = torch.linspace(0, nq - 1, n, device="cuda").long()
    return xq, pick


def flat_10m_inputs(torch):
    """configs[1]: xb [10M, 128], xq [10k, 128] and the indices of the 64 sampled queries"""
    N, d, nq = 10_000_000, 128, 10_000
    xb = _rows(torch, N, d, 1234)
    xq, pick = _sample_queries(torch, nq, d, 1235)
    return xb, xq, pick


def ivfflat_10m_index(torch, fb, res):
    """configs[2]: GpuIndexIVFFlat N=10M nlist=4096 nprobe=64.  The coarse centroids are seeded uniform rows (the
    random-sample start of k-means) rather than a device k-means result: float atomics make the latter vary in the
    last bits from run to run, and the stored reference answers are only valid for one exact index content."""
    N, d, nlist, nprobe = 10_000_000, 128, 4096, 64
    idx = fb.GpuIndexIVFFlat(res, d, nlist, fb.METRIC_L2)
    idx.setCoarseCentroids(_rows(torch, nlist, d, 4321).cpu().numpy())
    idx.setIsTrained(True)
    idx.reserveMemory(N + N // 8)
    for c0 in range(0, N, 1_000_000):
        idx.add(_rows(torch, 1_000_000, d, 1234 + c0 // 1_000_000))
    idx.nprobe = nprobe
    return idx


def sampled_pq_codebooks(torch, cent, M):
    """PQ codebooks [M, 256, d/M] cut from the residuals of 256 seeded uniform rows to their nearest coarse centroid (the
    random-sample start of PQ training): reproducible for the reason given in ivfflat_10m_index"""
    x = _rows(torch, 256, cent.shape[1], 4322).double()
    c = cent.double()
    a = ((x * x).sum(1, keepdim=True) - 2 * x @ c.T + (c * c).sum(1)).argmin(dim=1)
    r = (x - c[a]).float()
    return r.reshape(256, M, -1).permute(1, 0, 2).contiguous().cpu().numpy()


def ivfpq_100m_index(torch, fb, res):
    """configs[3]: GpuIndexIVFPQ N=100M nlist=4096 M=32 nprobe=32 over seeded uniform coarse centroids (see
    ivfflat_10m_index) and sampled_pq_codebooks"""
    N, d, nlist, M, nprobe = 100_000_000, 128, 4096, 32, 32
    idx = fb.GpuIndexIVFPQ(res, d, nlist, M, 8, fb.METRIC_L2)
    cent = _rows(torch, nlist, d, 4321)
    idx.setCoarseCentroids(cent.cpu().numpy())
    idx.setPQCentroids(sampled_pq_codebooks(torch, cent, M))
    idx.setIsTrained(True)
    idx.reserveMemory(N + N // 8)
    CH = 2_000_000
    for c0 in range(0, N, CH):
        idx.add(_rows(torch, CH, d, 1234 + c0 // CH, chunk=CH))
    idx.nprobe = nprobe
    return idx


def test_flat_l2_10m_vs_reference(res, ref_outputs_fullsize):
    """configs[1] vs faiss::knn_L2sqr over all 10M rows: uniform floats -> compareLists semantics with distances
    <= 1e-4 relative; integer-valued rows -> distances bit-exact and ids exact up to the tie group at rank k."""
    import torch

    import faiss_b200 as fb
    from oracle import oracle_np as o

    d, k = 128, 100
    xb, xq, pick = flat_10m_inputs(torch)
    idx = fb.GpuIndexFlatL2(res, d)
    idx.add(xb)
    D, I = idx.search(xq, k)  # the full nq=10k batch: the schedule the bench runs
    assert idx.lastSearchInfo()["tensor_cores"] == 1
    rD, rI = ref_outputs_fullsize["flat_D"], ref_outputs_fullsize["flat_I"]
    gD, gI = D[pick].cpu().numpy(), I[pick].cpu().numpy()
    st = o.compare_lists(rD, rI, gD, gI, eps=1e-4, pct_max_diff1=0.01, pct_max_diffN=0.005)
    assert (rI == gI).mean() > 0.97, st
    assert np.max(np.abs(rD - gD) / np.maximum(rD, 1e-20)) <= 1e-4
    # ---- integer regime at full size: every product and partial sum is exact in fp16 / fp32
    del idx
    xbi = torch.floor(xb * 16)
    del xb
    xqi = torch.floor(xq * 16)
    idx = fb.GpuIndexFlatL2(res, d)
    idx.add(xbi)
    D, I = idx.search(xqi, k)
    assert idx.lastSearchInfo()["tensor_cores"] == 1
    rD, rI = ref_outputs_fullsize["flatint_D"], ref_outputs_fullsize["flatint_I"]
    gD, gI = D[pick].cpu().numpy(), I[pick].cpu().numpy()
    assert np.array_equal(rD, gD), "integer regime: distances must be bit-exact"
    for q in range(len(pick)):
        inner = gD[q] < gD[q, k - 1]  # below the rank-k tie group both sides hold exactly the same ids
        assert set(gI[q][inner].tolist()) == set(rI[q][rD[q] < rD[q, k - 1]].tolist())
        # our order inside equal distances is ascending id (the CPU result handlers' rule)
        same = gD[q, 1:] == gD[q, :-1]
        assert (gI[q, 1:][same] > gI[q, :-1][same]).all()


def test_ivfflat_10m_vs_reference(res, ref_outputs_fullsize):
    """configs[2]: GpuIndexIVFFlat N=10M nlist=4096 nprobe=64 k=100 vs faiss::IndexIVFFlat holding the same
    centroids and the same inverted lists (pulled with getListVectorData / getListIndices)."""
    import torch

    import faiss_b200 as fb
    from oracle import oracle_np as o

    N, d, nlist, nq, k = 10_000_000, 128, 4096, 10_000, 100
    idx = ivfflat_10m_index(torch, fb, res)
    assert idx.ntotal == N
    assert sum(idx.getListLength(l) for l in range(nlist)) == N
    xq, pick = _sample_queries(torch, nq, d, 1235)
    D, I = idx.search(xq, k)
    rD, rI = ref_outputs_fullsize["ivfflat_D"], ref_outputs_fullsize["ivfflat_I"]
    gD, gI = D[pick].cpu().numpy(), I[pick].cpu().numpy()
    o.compare_lists(rD, rI, gD, gI, eps=1e-4, pct_max_diff1=0.02, pct_max_diffN=0.01)
    assert (rI == gI).mean() > 0.95


def test_ivfpq_100m_vs_reference(res, ref_outputs_fullsize):
    """configs[3]: GpuIndexIVFPQ N=100M nlist=4096 M=32 nprobe=32 k=100 vs faiss::IndexIVFPQ holding the same
    coarse centroids, PQ codebooks and list bytes (the clone direction of BASELINE.md section 3.4)."""
    import torch

    import faiss_b200 as fb
    from oracle import oracle_np as o

    N, d, nq, k = 100_000_000, 128, 10_000, 100
    idx = ivfpq_100m_index(torch, fb, res)
    assert idx.ntotal == N
    xq, pick = _sample_queries(torch, nq, d, 1235)
    D, I = idx.search(xq, k)
    rD, rI = ref_outputs_fullsize["ivfpq_D"], ref_outputs_fullsize["ivfpq_I"]
    gD, gI = D[pick].cpu().numpy(), I[pick].cpu().numpy()
    # PQ distances of 100M codes have many near-ties at rank ~100: ids may swap between adjacent ranks,
    # distances agree to fp32 summation order (the reference test's own tolerance is 0.035 / 0.1 / 0.06)
    o.compare_lists(rD, rI, gD, gI, eps=2e-4, pct_max_diff1=0.03, pct_max_diffN=0.015)
    assert np.max(np.abs(rD - gD) / np.maximum(rD, 1e-20)) <= 2e-4
