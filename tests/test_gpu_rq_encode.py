"""RQ encode parity: CUDA path (through the C ABI) vs the oracle and the reference's golden codes.
Bar: bit-exact int32 codes, except rows whose top-2 distance gap is below the stated fp32 epsilon
(oracle.TIE_EPS_DEFAULT = 2^-20 relative); such ties are counted and bounded."""
import numpy as np
import pytest
import torch

from oracle import oracle
from gpu_util import ctx, dev, tensor_modes

pytestmark = pytest.mark.gpu


def _check(X, cb, codes_gpu, codes_ref, max_tie_frac=2e-3, metric="l2"):
    rep = oracle.classify_code_mismatches(X, cb, codes_ref, codes_gpu, dist_mode=metric)
    assert rep["n_hard"] == 0, f"hard mismatches: {rep['hard_rows'][:8]} worst gap {rep['worst_rel_gap']:.3e}"
    assert rep["n_ties"] <= max(1, int(max_tie_frac * len(X))), rep
    return rep


def test_golden_codes(case):
    c = ctx()
    for mode in tensor_modes(c, case.d, case.M, case.K):
        codes = c.rq_encode(dev(case.X), dev(case.codebook), mode=mode).cpu().numpy()
        assert codes.dtype == np.int32
        rep = _check(case.X, case.codebook, codes, case.codes)
        print(case.name, mode, "ties", rep["n_ties"])


def test_golden_codes_ip_metric(case):
    c = ctx()
    codes = c.rq_encode(dev(case.X), dev(case.codebook), metric="ip", mode="exact").cpu().numpy()
    _check(case.X, case.codebook, codes, case.codes_ip, metric="ip")


def test_residual_output_matches_reference_arithmetic(gauss):
    c = ctx()
    X, cb = gauss.X, gauss.codebook
    res = torch.empty((gauss.n, gauss.d), device="cuda:0")
    codes = c.rq_encode(dev(X), dev(cb), mode="exact", residual=res).cpu().numpy()
    ref_codes, ref_res = oracle.rq_encode(X, cb, return_residual=True)
    same = (codes == ref_codes).all(1)
    assert same.mean() > 0.99
    # fp32 elementwise subtraction in the same order as pq.py:304-305 -> bit-identical residual
    assert np.array_equal(res.cpu().numpy()[same], ref_res[same])


@pytest.mark.parametrize("n", [0, 1, 3, 31, 33, 127, 129, 1000])
def test_ragged_sizes(gauss, n):
    c = ctx()
    X = gauss.X[:n]
    for mode in tensor_modes(c, gauss.d, gauss.M, gauss.K):
        codes = c.rq_encode(dev(X) if n else torch.empty((0, gauss.d), device="cuda:0"), dev(gauss.codebook), mode=mode)
        assert tuple(codes.shape) == (n, gauss.M)
        if n:
            _check(X, gauss.codebook, codes.cpu().numpy(), gauss.codes[:n], max_tie_frac=1.0)


def test_duplicate_centroids_lowest_index_wins():
    c = ctx()
    rs = np.random.RandomState(0)
    X = rs.standard_normal((512, 64)).astype(np.float32)
    cb = rs.standard_normal((2, 16, 64)).astype(np.float32)
    cb[0, 11] = cb[0, 2]
    codes = c.rq_encode(dev(X), dev(cb), mode="exact").cpu().numpy()
    assert not (codes[:, 0] == 11).any()
    assert (codes == oracle.rq_encode(X, cb)).all()


def test_host_buffer_variant_streams_chunks(gauss):
    c = ctx()
    codes = np.empty((gauss.n, gauss.M), dtype=np.int32)
    stats = c.rq_encode_host(gauss.X, gauss.codebook, codes, mode="auto", chunk_rows=700)  # ragged last chunk
    assert stats[1] == gauss.n
    _check(gauss.X, gauss.codebook, codes, gauss.codes)


def test_larger_random_against_oracle():
    c = ctx()
    rs = np.random.RandomState(11)
    n, d, M, K = 60000, 768, 4, 32
    X = rs.standard_normal((n, d)).astype(np.float32)
    # a codebook with reference-like statistics: level means of random subsets of the residual
    cb = np.empty((M, K, d), dtype=np.float32)
    res = X.copy()
    for j in range(M):
        lab = rs.randint(0, K, size=n)
        for k in range(K):
            cb[j, k] = res[lab == k][:400].mean(0)
        res = res - cb[j][oracle.rq_encode(res, cb[j : j + 1])[:, 0]]
    ref = oracle.rq_encode(X, cb, batch_size=1024)
    for mode in tensor_modes(c, d, M, K):
        codes, stats = c.rq_encode(dev(X), dev(cb), mode=mode, return_stats=True)
        rep = _check(X, cb, codes.cpu().numpy(), ref)
        print(mode, "ties", rep["n_ties"], "flagged", int(stats[0]), "rows", int(stats[1]))
        assert int(stats[1]) == n


def test_pq_dropin_get_document_cluster(gauss, tmp_path):
    """The reference-shaped entry point end to end: ProductQuantization.initialize (from the
    reference's own .pt file) + get_document_cluster on a numpy array -> same dictionaries."""
    import os

    from mevi_b200.pq import ProductQuantization

    pq = ProductQuantization("rq", gauss.M, 5, "l2", gauss.d, "kmeans", "grad")
    pq.initialize(os.path.join(gauss.dir, "codebook.pt"), gauss.X, 0, 41, None, 1024)
    assert not pq.get_preds
    clus, mapping = pq.get_document_cluster(gauss.X, 0, 1, 128, True)
    codes = np.array([mapping[i] for i in range(gauss.n)], dtype=np.int32)
    rep = _check(gauss.X, gauss.codebook, codes, gauss.codes)
    if rep["n_mismatch"] == 0:
        assert clus == gauss.pickle("rqclus.pkl") and mapping == gauss.pickle("rqmapping.pkl")
        assert list(clus.keys()) == list(gauss.pickle("rqclus.pkl").keys())
    # 2-rank row-block sharding, merged like LogPklFile (main_models.py:289-310)
    merged = {}
    for r in range(2):
        cdict = pq.get_document_cluster(gauss.X, r, 2, 128, False)
        for k, v in cdict.items():
            merged.setdefault(k, []).extend(v)
    assert merged == clus


@pytest.mark.parametrize("n,d,M,K,metric", [(5000, 128, 2, 64, "l2"), (4099, 1024, 3, 32, "l2"), (6000, 64, 4, 32, "l2"),
                                            (5000, 256, 1, 128, "l2"), (5000, 768, 4, 32, "ip"), (3000, 320, 2, 32, "l2"),
                                            (3000, 100, 2, 8, "l2")])
def test_shape_family_tensor_and_exact(n, d, M, K, metric):
    """Other members of the shape family (levels, codebook sizes, widths, metric): whichever modes the
    library supports for the shape must agree with the oracle; 'auto' must always work."""
    c = ctx()
    rs = np.random.RandomState(d + M + K)
    centers = rs.standard_normal((K, d)).astype(np.float32)
    X = (centers[rs.randint(0, K, n)] + 0.7 * rs.standard_normal((n, d))).astype(np.float32)
    cb = np.empty((M, K, d), dtype=np.float32)
    res = X.copy()
    for j in range(M):
        cb[j] = res[rs.choice(n, K, replace=False)] * (0.9 if j == 0 else 0.5)
        res = res - cb[j][oracle.rq_encode(res, cb[j : j + 1], dist_mode=metric)[:, 0]]
    ref = oracle.rq_encode(X, cb, dist_mode=metric)
    modes = tensor_modes(c, d, M, K, metric) + ["auto"]
    for mode in modes:
        codes, stats = c.rq_encode(dev(X), dev(cb), metric=metric, mode=mode, return_stats=True)
        rep = _check(X, cb, codes.cpu().numpy(), ref, metric=metric)
        print(f"d={d} M={M} K={K} {metric} {mode}: ties {rep['n_ties']} flagged {int(stats[0])}")


def test_badly_scaled_and_outlier_rows_still_exact(gauss):
    """Rows far outside the sampled range (fp16 overflow after scaling) and all-zero rows must come out
    right: the tensor path sends them to the exact kernel instead of trusting the prefilter."""
    c = ctx()
    X = gauss.X[:8192].copy()
    X[7] *= 1e6
    X[100] = 0.0
    X[200] *= 1e-6
    X[4000:4010] *= 3e4
    ref = oracle.rq_encode(X, gauss.codebook)
    for mode in tensor_modes(c, gauss.d, gauss.M, gauss.K):
        codes = c.rq_encode(dev(X), dev(gauss.codebook), mode=mode).cpu().numpy()
        _check(X, gauss.codebook, codes, ref)


def test_config_i_100k_golden_codes():
    """BASELINE.json configs[0] (100k x 768, reference-built codebook): every kernel mode against the reference's codes."""
    import json
    import os

    import datasets
    from conftest import GOLDEN

    d = os.path.join(GOLDEN, "gauss100k")
    meta = json.load(open(os.path.join(d, "meta.json")))
    X = datasets.case_docs("gauss100k")
    assert datasets.sha256(X) == meta["x_sha256"]
    cb = torch.load(os.path.join(d, "codebook.pt"), map_location="cpu", weights_only=False).detach().numpy()
    want = np.load(os.path.join(d, "codes_u8.npy")).astype(np.int32)
    c = ctx()
    for mode in tensor_modes(c, 768, 4, 32):
        codes, stats = c.rq_encode(dev(X), dev(cb), mode=mode, return_stats=True)
        rep = _check(X, cb, codes.cpu().numpy(), want)
        print("gauss100k", mode, "mismatch", rep["n_mismatch"], "ties", rep["n_ties"], "stats", stats.tolist()[:3])
