"""Pins the numpy oracle (oracle/oracle_np.py) against the reference: golden fixtures generated
from the unmodified reference CPU library (tests/golden/make_golden.py and
tests/golden/make_reference_outputs.py).  No GPU needed."""
import numpy as np
import pytest

from oracle import oracle_np as o


def test_float_rand_matches_reference_bits(golden):
    assert np.array_equal(o.float_rand(5000, 1234), golden["float_rand_5000_s1234"])
    assert np.array_equal(o.float_rand(300, 7), golden["float_rand_300_s7"])


def test_rand_perm_matches_reference(golden):
    assert np.array_equal(o.rand_perm(1000, 42), golden["rand_perm_1000_s42"])


def _flat_inputs(golden):
    N, d, nq, k = golden["flat_shape"]
    xb = o.float_rand(N * d, 1234).reshape(N, d)
    xq = o.float_rand(nq * d, 1235).reshape(nq, d)
    return xb, xq, int(k)


@pytest.mark.parametrize("metric,name", [(1, "l2"), (0, "ip")])
def test_flat_oracle_vs_golden(golden, metric, name):
    xb, xq, k = _flat_inputs(golden)
    D, I = o.knn_flat(xq, xb, k, metric)
    gD, gI = golden["flat_%s_D" % name], golden["flat_%s_I" % name]
    # uniform floats: ids agree except where fp32 rounding swaps near-ties; distances to 1e-4 rel
    assert (I == gI).mean() > 0.99
    o.compare_lists(gD, gI, D, I, eps=1e-4, pct_max_diff1=0.01, pct_max_diffN=0.005)


@pytest.mark.parametrize("k", [10, 100])
def test_flat_integer_regime_ids_exact(golden, k):
    """values in {0..15}, d=64: every product and partial sum is exact in fp32, so the reference's
    ids (heap handler for k<100, reservoir for k>=100) are reproduced bit for bit by the
    (distance asc, id asc) rule."""
    N, d, nq = golden["flatint_shape"]
    xb = np.floor(o.float_rand(N * d, 11).reshape(N, d) * 16).astype(np.float32)
    xq = np.floor(o.float_rand(nq * d, 12).reshape(nq, d) * 16).astype(np.float32)
    D, I = o.knn_flat(xq, xb, k, 1)
    assert np.array_equal(D, golden["flatint_l2_k%d_D" % k])
    assert np.array_equal(I, golden["flatint_l2_k%d_I" % k])


def test_merge_vs_golden(golden):
    D, I = o.merge_knn_results(golden["merge_allD"], golden["merge_allI"], 1)
    assert np.array_equal(I, golden["merge_I"])
    assert np.array_equal(D, golden["merge_D"])


def _ivfpq_fixture(golden, name):
    N, d, nlist, M, nq, k, nprobe = [int(v) for v in golden["ivfpq_shape"]]
    lens = golden["ivfpq_%s_lens" % name]
    codes_all = golden["ivfpq_%s_codes" % name]
    ids_all = golden["ivfpq_%s_ids" % name]
    codes, ids = [], []
    c0 = i0 = 0
    for n in lens:
        codes.append(codes_all[c0 : c0 + n * M])
        ids.append(ids_all[i0 : i0 + n])
        c0 += n * M
        i0 += n
    xb = o.float_rand(N * d, 21).reshape(N, d)
    xq = o.float_rand(nq * d, 22).reshape(nq, d)
    return dict(N=N, d=d, nlist=nlist, M=M, nq=nq, k=k, nprobe=nprobe, xb=xb, xq=xq, codes=codes, ids=ids,
                centroids=golden["ivfpq_%s_centroids" % name], pq=golden["ivfpq_%s_pq" % name],
                D=golden["ivfpq_%s_D" % name], I=golden["ivfpq_%s_I" % name])


@pytest.mark.parametrize("metric,name", [(1, "l2"), (0, "ip")])
def test_ivfpq_search_oracle_vs_golden(golden, metric, name):
    f = _ivfpq_fixture(golden, name)
    D, I = o.ivfpq_search(f["xq"], f["k"], f["nprobe"], f["centroids"], f["pq"], f["codes"], f["ids"], metric)
    o.compare_lists(f["D"], f["I"], D, I, eps=2e-4, pct_max_diff1=0.02, pct_max_diffN=0.01)


def test_pq_encode_oracle_vs_golden_lists(golden):
    """the codes the reference stored are reproduced by assign -> residual -> pq_encode"""
    f = _ivfpq_fixture(golden, "l2")
    a = o.ivf_assign(f["xb"], f["centroids"], 1)
    codes = o.pq_encode(f["xb"] - f["centroids"][a], f["pq"])
    stored = {}
    for l in range(f["nlist"]):
        for c, i in zip(f["codes"][l].reshape(-1, f["M"]), f["ids"][l]):
            stored[int(i)] = (l, c)
    mism = sum(1 for i in range(f["N"]) if stored[i][0] != a[i] or (stored[i][1] != codes[i]).any())
    assert mism <= f["N"] * 0.002  # fp near-ties only


def test_kmeans_oracle_vs_golden(golden):
    x = o.float_rand(5000 * 8, 31).reshape(5000, 8)
    cent, obj = o.kmeans(x, 20, niter=8, seed=123)
    assert np.allclose(obj, golden["kmeans_obj"], rtol=1e-4)
    assert np.allclose(cent, golden["kmeans_centroids"], rtol=1e-3, atol=1e-4)
    cent, obj = o.kmeans(x, 4, niter=5, seed=99, max_points_per_centroid=256)
    assert np.allclose(obj, golden["kmeans_sub_obj"], rtol=1e-4)
    assert np.allclose(cent, golden["kmeans_sub_centroids"], rtol=1e-3, atol=1e-4)


def test_ivfflat_search_oracle_vs_golden(golden):
    """pins oracle_np.ivfflat_search on the reference's own IndexIVFFlat lists, centroids and results
    (fixture minted by tests/golden/make_golden.py from oracle/_ref)"""
    N, d, nlist, M, nq, k, nprobe = [int(v) for v in golden["ivfpq_shape"]]
    xb = o.float_rand(N * d, 21).reshape(N, d)
    xq = o.float_rand(nq * d, 22).reshape(nq, d)
    lens, ids_all = golden["ivfflat_lens"], golden["ivfflat_ids"]
    assert lens.sum() == N
    vecs, ids = [], []
    i0 = 0
    for n in lens:
        li = ids_all[i0 : i0 + n]
        ids.append(li)
        vecs.append(xb[li])
        i0 += n
    D, I = o.ivfflat_search(xq, k, nprobe, golden["ivfflat_centroids"], vecs, ids, 1)
    o.compare_lists(golden["ivfflat_D"], golden["ivfflat_I"], D, I, eps=1e-4, pct_max_diff1=0.01, pct_max_diffN=0.005)
    # and the assignment that produced those lists is the oracle's coarse assignment (up to near-ties)
    a = o.ivf_assign(xb, golden["ivfflat_centroids"], 1)
    owner = np.empty(N, dtype=np.int64)
    i0 = 0
    for l, n in enumerate(lens):
        owner[ids_all[i0 : i0 + n]] = l
        i0 += n
    assert (a != owner).sum() <= N * 0.002


def test_pq_train_oracle_vs_golden(golden):
    """ProductQuantizer::train (M independent k-means, same seeds) reproduced by the numpy restatement"""
    n, d, M, niter, seed = [int(v) for v in golden["pqtrain_shape"]]
    x = o.float_rand(n * d, 41).reshape(n, d)
    c = o.pq_train(x, M, niter=niter, seed=seed)
    assert np.allclose(c, golden["pqtrain_centroids"], rtol=1e-3, atol=1e-4)


def test_kmeans_spherical_ip_oracle_vs_golden(golden):
    """Clustering(spherical=True) over an inner-product index (GpuIndexIVF.cu:72-76 for METRIC_INNER_PRODUCT)"""
    x = o.float_rand(3000 * 8, 51).reshape(3000, 8) - np.float32(0.5)
    cent, obj = o.kmeans(x, 12, niter=6, seed=77, metric=0, spherical=True)
    assert np.allclose(obj, golden["kmeans_sph_obj"][: len(obj)], rtol=1e-4)
    assert np.allclose(cent, golden["kmeans_sph_centroids"], rtol=1e-3, atol=1e-4)
    assert np.allclose(np.linalg.norm(cent, axis=1), 1.0, atol=1e-5)


# ------------------------------------------------------------------ checks against the reference library's own answers
# (stored by tests/golden/make_reference_outputs.py from oracle/_ref; the inputs are regenerated here from the same seeds)
FLAT_LIVE_CASES = [(2000, 16, 30, 5, 1), (1500, 40, 11, 120, 0), (50, 8, 4, 60, 1)]


def flat_live_inputs():
    """(xb, xq, k, metric) per FLAT_LIVE_CASES entry"""
    rs = np.random.RandomState(0)
    for (N, d, nq, k, metric) in FLAT_LIVE_CASES:
        xb = rs.rand(N, d).astype(np.float32)
        xq = rs.rand(nq, d).astype(np.float32)
        yield xb, xq, k, metric


def precomputed_onoff_inputs():
    """xb, xq of test_precomputed_table_on_off_same_ids: IndexIVFPQ(d=16, nlist=8, M=4), niter 4, nprobe 3, k 10"""
    rs = np.random.RandomState(1)
    xb = rs.rand(4000, 16).astype(np.float32)
    xq = rs.rand(20, 16).astype(np.float32)
    return xb, xq


def precomputed_form_inputs():
    """xb, xq of test_oracle_precomputed_form_vs_reference: IndexIVFPQ(d=32, nlist=16, M=8), niter 4, nprobe 4, k 10"""
    rs = np.random.RandomState(7)
    xb = rs.rand(6000, 32).astype(np.float32)
    xq = rs.rand(30, 32).astype(np.float32)
    return xb, xq


def stored_lists(outputs, prefix, xb):
    """per-list codes and ids of a reference IndexIVFPQ stored by make_reference_outputs.py: the oracle's encoding of each
    vector's residual to its stored list, with the stored codes where the reference's differ (fp near-ties)"""
    cent, pq, a = outputs[prefix + "_centroids"], outputs[prefix + "_pq"], outputs[prefix + "_list"].astype(np.int64)
    rows = outputs[prefix + "_patch_rows"]
    assert rows.size <= xb.shape[0] * 0.002  # the restatement of compute_code agrees but for near-ties
    codes = o.pq_encode(xb - cent[a], pq)
    codes[rows] = outputs[prefix + "_patch_codes"]
    li = [np.flatnonzero(a == l) for l in range(cent.shape[0])]
    return [codes[i].reshape(-1) for i in li], li


def test_flat_vs_reference_live(ref_outputs):
    for i, (xb, xq, k, metric) in enumerate(flat_live_inputs()):
        rD, rI = ref_outputs["flat_%d_D" % i], ref_outputs["flat_%d_I" % i]
        D, I = o.knn_flat(xq, xb, k, metric)
        o.compare_lists(rD, rI, D, I, eps=1e-4, pct_max_diff1=0.02, pct_max_diffN=0.01)


def test_precomputed_table_on_off_same_ids(ref_outputs):
    """tests/test_index_accuracy.py:506-508: precomputed table on/off gives identical ids; the
    oracle's residual form is therefore a faithful restatement of either mode."""
    xb, xq = precomputed_onoff_inputs()
    D1, I1 = ref_outputs["onoff_D1"], ref_outputs["onoff_I1"]
    D0, I0 = ref_outputs["onoff_D0"], ref_outputs["onoff_I0"]
    assert (I0 == I1).mean() > 0.98
    assert np.allclose(D0, D1, rtol=1e-4, atol=1e-5)
    # the stored index is the one the reference trained on these inputs: the oracle reproduces its lists and answers
    cent, pq = ref_outputs["onoff_centroids"], ref_outputs["onoff_pq"]
    lc, li = stored_lists(ref_outputs, "onoff", xb)
    D, I = o.ivfpq_search(xq, 10, 3, cent, pq, lc, li, 1, precomputed=False)
    o.compare_lists(D0, I0, D, I, eps=1e-4, pct_max_diff1=0.02, pct_max_diffN=0.01)


def test_oracle_precomputed_form_vs_reference(ref_outputs):
    """the numpy restatement of the precomputed-table decomposition (what the GPU scan evaluates when
    usePrecomputedTables is active) against the reference CPU index with use_precomputed_table = 1, and
    against the residual form: same ids up to near-ties, distances within 1e-4 relative"""
    xb, xq = precomputed_form_inputs()
    k, nprobe = 10, 4
    rD, rI = ref_outputs["pcform_D"], ref_outputs["pcform_I"]
    cent, pq = ref_outputs["pcform_centroids"], ref_outputs["pcform_pq"]
    lc, li = stored_lists(ref_outputs, "pcform", xb)
    D1, I1 = o.ivfpq_search(xq, k, nprobe, cent, pq, lc, li, 1, precomputed=True)
    D0, I0 = o.ivfpq_search(xq, k, nprobe, cent, pq, lc, li, 1, precomputed=False)
    o.compare_lists(rD, rI, D1, I1, eps=1e-4, pct_max_diff1=0.02, pct_max_diffN=0.01)
    o.compare_lists(D0, I0, D1, I1, eps=1e-4, pct_max_diff1=0.02, pct_max_diffN=0.01)
