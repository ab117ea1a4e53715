"""CPU self-tests of the boundary generators of test_gpu_prefilter_bounds.py: they must put decisions where they claim,
and the float64 quantities they return must be the ones a fresh float64 computation gives."""
import numpy as np
import pytest

from oracle import oracle
from test_gpu_prefilter_bounds import (RQ_REGIMES, TIE, adversarial_rounding_docs, assert_boundary_coverage, check_topk_float64,
                                       decided_gaps, fp32_dot_bound, pq_gap_rows, pq_path64, rq_boundary_set, rq_path64,
                                       topk_boundary_docs)


@pytest.mark.parametrize("regime", ["gauss", "gauss_ip", "offset", "mixed_norms", "clustered_M2_K32"])
def test_rq_generator_sits_on_the_bound(regime):
    X, cb, metric, lev, c64, rel = rq_boundary_set(regime)
    assert X.dtype == np.float32 and len(X) > 0.9 * (6000 if regime.startswith("clustered") else 8000)
    g = decided_gaps(rel, lev)
    assert_boundary_coverage(g, near_frac=0.15 if regime == "mixed_norms" else 0.2)
    assert (g >= 0).all() and (g < 2.0 ** -6).mean() > 0.9
    codes, rel2, _ = rq_path64(X, cb, metric)  # returned quantities = a fresh float64 path of the returned rows
    assert np.array_equal(codes, c64) and np.array_equal(rel, rel2)
    # the float64 codes agree with the reference encoder up to ties of the oracle's own rule
    ref = oracle.rq_encode(X[:1500], cb, dist_mode=metric, batch_size=1024)
    rep = oracle.classify_code_mismatches(X[:1500], cb, c64[:1500], ref, dist_mode=metric)
    assert rep["n_hard"] == 0


def test_rq_regime_list_is_built():
    assert {"gauss", "offset", "mixed_norms"} <= set(RQ_REGIMES)
    X, cb, metric, lev, _, _ = rq_boundary_set("mixed_norms")
    norms = np.linalg.norm(X, axis=1)
    assert norms.min() < 2.0 ** -15 and norms.max() > 2.0 ** 12 and (lev == 0).all() and metric == "ip"
    X, cb, _, _, _, _ = rq_boundary_set("offset")
    mu = X.mean(0)
    assert np.linalg.norm(mu) >= 10 * np.sqrt(((X - mu) ** 2).sum(1).mean()) * 0.9


@pytest.mark.parametrize("metric", ["l2", "ip"])
def test_pq_generator_sits_on_the_bound(metric):
    rs = np.random.RandomState(1)
    M, K, ds = 8, 64, 32
    X = rs.standard_normal((3000, M * ds)).astype(np.float32)
    cb = (rs.standard_normal((M, K, ds)) * 0.7).astype(np.float32)
    Xn, dl, c64, rel = pq_gap_rows(X, cb, rs, metric)
    assert_boundary_coverage(rel.ravel())
    codes, rel2, _ = pq_path64(Xn, cb, metric)
    assert np.array_equal(codes, c64) and np.array_equal(rel, rel2)
    ties, real = oracle.classify_pq_mismatches(Xn, cb, oracle.pq_encode(Xn, cb, metric), c64, metric)
    assert real == 0


def test_topk_generator_and_checker():
    rs = np.random.RandomState(2)
    n, d, nq, k = 4000, 64, 3, 50
    D = rs.standard_normal((n, d)).astype(np.float32)
    Q = rs.standard_normal((nq, d)).astype(np.float32)
    D2, rel, picks = topk_boundary_docs(D, Q, k, rs)
    assert (np.abs(rel) < TIE).mean() > 0.05 and (np.abs(rel) < 2.0 ** -5).all()
    assert ((rel > 0).mean(1) > 0.3).all() and ((rel < 0).mean(1) > 0.3).all()
    # the float64 answer passes the checker; dropping a true member for the (k+1)-th document fails it unless tied
    S = Q.astype(np.float64) @ D2.astype(np.float64).T
    ids = np.argsort(-S, axis=1, kind="stable")[:, :k]
    sc = np.take_along_axis(S, ids, 1).astype(np.float32)
    check_topk_float64(sc, ids, Q, D2, k)
    order = np.argsort(-S[0], kind="stable")
    far = next(p for p in range(k, n) if S[0, order[k - 1]] - S[0, order[p]] > 1e-3)
    bad = ids.copy()
    bad[0, k - 1] = order[far]
    sc_bad = sc.copy()
    sc_bad[0, k - 1] = np.float32(S[0, order[far]])
    with pytest.raises(AssertionError):
        check_topk_float64(sc_bad, bad, Q, D2, k)


def test_adversarial_rounding_docs_need_the_full_margin():
    """emulated fp16 prefilter: the weakest members sit > margin/8 below the k-th approximate score, < margin/2"""
    D, q, members = adversarial_rounding_docs()
    k, d = len(members), D.shape[1]
    exact = D.astype(np.float64) @ q[0].astype(np.float64)
    assert set(np.argsort(-exact, kind="stable")[:k].tolist()) == set(members.tolist())
    approx = (D * 2048.0).astype(np.float16).astype(np.float64).sum(1)  # scale 2^11, query image exact
    dmax = np.linalg.norm(D.astype(np.float64), axis=1).max() * 2048.0
    e_rel = 1.01 * 2.0 ** -10 * np.sqrt(d) * dmax                      # the relative term of the margin, per side
    shortfall = np.sort(approx)[-k] - approx[members].min()
    assert e_rel / 4 < shortfall < e_rel
    rival_best = np.sort(np.delete(exact, members))[-1]
    assert exact[members].min() - rival_best > 2 * fp32_dot_bound(q, D[members]).max()
