"""Top-k re-rank of a multi-cluster index (`--doc_multiclus > 1`, main_models.py:3998-4011 + the sort and the
`[:save_hard_neg]` truncation): `ClusterReranker.rerank(..., multiclus_score_aggr=...)` and the occurrence table."""
import os
import pickle
from collections import Counter

import numpy as np
import pytest
import torch

from oracle import oracle
from gpu_util import dev

pytestmark = pytest.mark.gpu


def _golden(case_name, what):
    from conftest import GOLDEN

    with open(os.path.join(GOLDEN, "rerank", f"{case_name}_{what}.pkl"), "rb") as fr:
        return pickle.load(fr)


def _reranker(X, clus, K):
    from mevi_b200.rerank import ClusterIndex, ClusterReranker

    return ClusterReranker(dev(X), ClusterIndex.from_cluster_dict(clus, K), mode="stream")


def _line_scores(text, q):
    """Scores field of the reference's hn line of query q (main_models.py:4046-4053)."""
    field = text.rstrip("\n").split("\n")[q].split("\t")[3]
    return np.asarray([float(v) for v in field.split(",")] if field else [], dtype=np.float64)


def _multiplicity(clus, dec_q):
    """document -> number of positions of the leaf list dec_q whose leaf lists it."""
    c = Counter()
    for leaf in dec_q:
        c.update(clus.get(tuple(int(v) for v in leaf), ()))
    return c


def _synthetic(nq=24, n=20000, d=64, K=16, L=24, seed=0):
    """Every document listed under its own leaf (2 digits, K = 16) and a neighbouring one (last digit + 1..3); each query
    asks for runs of 4 neighbouring leaves, so it often holds both leaves of a document.  Query 0 has one leaf only
    (fewer candidates than the larger k)."""
    rs = np.random.RandomState(seed)
    X = rs.standard_normal((n, d)).astype(np.float32)
    Q = rs.standard_normal((nq, d)).astype(np.float32)
    code1 = rs.randint(0, K, size=(n, 2))
    code2 = code1.copy()
    code2[:, 1] = (code2[:, 1] + 1 + rs.randint(0, 3, n)) % K
    clus = {}
    for doc in range(n):
        for c in (code1[doc], code2[doc]):
            clus.setdefault((int(c[0]), int(c[1])), []).append(doc)
    dec = np.zeros((nq, L, 2), np.int64)
    for q in range(nq):
        first = rs.choice(K, L // 4, replace=False)
        start = rs.randint(0, K, L // 4)
        for j in range(L):
            dec[q, j] = (first[j // 4], (start[j // 4] + j % 4) % K)
    dec[0, 1:] = K  # codes outside [0, K): no such leaf
    return X, Q, clus, dec, K


def test_plain_rerank_on_a_multicluster_index_repeats_documents():
    """What `rerank()` without an aggregation returns on a --doc_multiclus 2 index: a document shared by two of the
    query's leaves is listed once per leaf, and its score is not the reference's 'add' score."""
    case_name, nb = "gauss768", 100
    from conftest import golden_case

    case = golden_case(case_name)
    dec = case.load(f"beam{nb}_labels.npy")
    mc = _golden(case_name, "multiclus_dict")
    fm = _golden(case_name, "multiclus_add")
    rr = _reranker(case.X, mc, case.K)
    s, i, n = (t.cpu().numpy() for t in rr.rerank(case.Q, dec, topk=200))
    n_rows_dup, n_dup, n_add_differs = 0, 0, 0
    for q in range(len(case.Q)):
        ids = i[q][i[q] >= 0]
        extra = len(ids) - len(set(ids.tolist()))
        n_rows_dup += extra > 0
        n_dup += extra
        want = dict(zip(fm["docs"][q], _line_scores(fm["lines"], q)))
        for p_, doc in enumerate(ids.tolist()):
            n_add_differs += abs(float(s[q, p_]) - want[doc]) > 1e-4
    print(f"plain rerank() on {case_name}_multiclus_dict: {n_rows_dup} of {len(case.Q)} queries list a document twice "
          f"({n_dup} extra entries); {n_add_differs} listed scores differ from the reference's 'add' score")
    assert n_rows_dup > 0 and n_dup > 0 and n_add_differs > 0


@pytest.mark.parametrize("aggr", ["add", "max"])
@pytest.mark.parametrize("case_name,nb", [("gauss768", 100), ("small64", 10)])
def test_topk_equals_the_executed_reference_loop(case_name, nb, aggr):
    """Against main_models.py:3912-4055 EXECUTED verbatim with doc_multiclus=2, save_hard_neg=200."""
    from conftest import golden_case

    case = golden_case(case_name)
    dec = case.load(f"beam{nb}_labels.npy")
    mc = _golden(case_name, "multiclus_dict")
    fm = _golden(case_name, f"multiclus_{aggr}")
    rr = _reranker(case.X, mc, case.K)
    s, i, n = (t.cpu().numpy() for t in rr.rerank(case.Q, dec, topk=200, multiclus_score_aggr=aggr))
    assert rr.last_path == "stream-multiclus"
    X64, Q64 = case.X.astype(np.float64), case.Q.astype(np.float64)
    for q in range(len(case.Q)):
        docs = fm["docs"][q][:200]
        kk = len(docs)
        want_s = _line_scores(fm["lines"], q)
        assert n[q] == fm["ndoc"][q]
        assert sorted(i[q, :kk].tolist()) == sorted(docs) and (i[q, kk:] == -1).all() and np.isneginf(s[q, kk:]).all()
        np.testing.assert_allclose(s[q, :kk], want_s, rtol=1e-5, atol=2e-4)
        mult = _multiplicity(mc, dec[q])
        agg64 = lambda doc: float(X64[doc] @ Q64[q]) * (mult[doc] if aggr == "add" else 1)
        for p_ in np.nonzero(i[q, :kk] != np.asarray(docs))[0]:  # order may differ only between (near-)equal scores
            assert abs(agg64(int(i[q, p_])) - agg64(int(docs[p_]))) <= 1e-4


@pytest.fixture(scope="module")
def synthetic():
    X, Q, clus, dec, K = _synthetic()
    rr = _reranker(X, clus, K)
    full = {aggr: tuple(t.cpu().numpy() for t in rr.rerank_all(Q, dec, multiclus_score_aggr=aggr)) for aggr in ("add", "max")}
    return X, Q, clus, dec, K, rr, full


def _assert_truncation_of_rerank_all(s, i, full, k, qs):
    off, ids_all, sc_all = full
    for r, q in enumerate(qs):
        a, b = off[q], off[q + 1]
        kk = min(k, b - a)
        assert np.array_equal(s[r, :kk], sc_all[a : a + kk]), f"query {q}: scores are not rerank_all's"
        assert np.array_equal(i[r, :kk], ids_all[a : a + kk]), f"query {q}: ids are not rerank_all's"
        assert np.isneginf(s[r, kk:]).all() and (i[r, kk:] == -1).all()
        assert len(set(i[r, :kk].tolist())) == kk


@pytest.mark.parametrize("aggr", ["add", "max"])
@pytest.mark.parametrize("k", [1, 10, 100, 1000, 2048])
def test_topk_equals_rerank_all_truncated(synthetic, k, aggr):
    X, Q, clus, dec, K, rr, full = synthetic
    s, i, n = (t.cpu().numpy() for t in rr.rerank(Q, dec, topk=k, multiclus_score_aggr=aggr))
    _assert_truncation_of_rerank_all(s, i, full[aggr], k, range(len(Q)))
    off = full[aggr][0]
    assert off[1] - off[0] < 1000 < (off[2:] - off[1:-1]).min()  # query 0 has fewer candidates than the larger k
    want_n = [sum(_multiplicity(clus, dec[q]).values()) for q in range(len(Q))]
    assert n.tolist() == want_n
    assert sum(want_n) > off[-1]  # documents did occur under several of a query's leaves


@pytest.mark.parametrize("aggr", ["add", "max"])
def test_splits_keep_one_entry_per_document(synthetic, aggr):
    """Two queries: each query's candidates are cut over many CTAs (splits); a document's occurrences fall into different
    splits, and exactly one of them may survive."""
    X, Q, clus, dec, K, rr, full = synthetic
    qs = [5, 9]
    s, i, n = (t.cpu().numpy() for t in rr.rerank(Q[qs], dec[qs], topk=100, multiclus_score_aggr=aggr))
    _assert_truncation_of_rerank_all(s, i, full[aggr], 100, qs)
    # a single huge leaf: its positions alone are spread over every split
    n_big = 30000
    rs = np.random.RandomState(3)
    Xb = rs.standard_normal((n_big, 64)).astype(np.float32)
    clus_b = {(0, 0): list(range(n_big)), (0, 1): list(range(0, n_big, 2)), (0, 2): list(range(0, n_big, 3))}
    dec_b = np.array([[[0, 2], [0, 0], [0, 1]]], np.int64)
    rrb = _reranker(Xb, clus_b, 4)
    sb, ib, nb = (t.cpu().numpy() for t in rrb.rerank(Xb[:1] * 0.5, dec_b, topk=100, multiclus_score_aggr=aggr))
    _assert_truncation_of_rerank_all(sb, ib, tuple(t.cpu().numpy() for t in rrb.rerank_all(Xb[:1] * 0.5, dec_b, aggr)), 100, [0])
    assert int(nb[0]) == n_big + n_big // 2 + (n_big + 2) // 3


def _exact_case():
    """Scores that are exact in fp32 whatever the summation order (one non-zero coordinate), so that the kernel and the
    oracle see the same s.  Leaves (M = 2, K = 4); the query's list repeats leaf (0, 0)."""
    d = 64
    s_of = {0: 1 + 2.0 ** -23, 1: 1 + 2.0 ** -22 + 2.0 ** -23, 2: 0.75, 3: -1.5, 4: -2.0, 5: 0.5, 6: 0.25}
    X = np.zeros((8, d), np.float32)
    for doc, v in s_of.items():
        X[doc, 0] = np.float32(v)
    X[7, 0] = np.float32(-0.125)
    A, B, Cl, D, E = (0, 0), (0, 1), (1, 2), (2, 3), (3, 0)
    clus = {A: [0, 1, 2, 5], B: [0, 1, 3], Cl: [0, 1, 6], D: [1, 7], E: [3, 4]}
    # doc 0: A x2, B, Cl -> c = 4 (3 distinct leaves, one repeated); doc 1: A x2, B, Cl, D -> c = 5; doc 2: A x2 -> c = 2
    dec = np.array([[A, B, A, Cl, D, E]], np.int64)
    Q = np.zeros((1, d), np.float32)
    Q[0, 0] = 1.0
    return X, Q, clus, dec


def test_add_is_the_fp32_fold_of_the_reference_with_multiplicities_above_two():
    X, Q, clus, dec = _exact_case()
    rr = _reranker(X, clus, 4)
    occ, n_occ = rr.index.occurrence_table()
    assert n_occ == 4  # document 1 is listed under four leaves
    for aggr in ("add", "max"):
        s, i, n = (t.cpu().numpy() for t in rr.rerank(Q, dec, topk=10, multiclus_score_aggr=aggr))
        (docs, scores, ndoc), = oracle.cluster_rerank(Q, X, clus, dec, multiclus_aggr=aggr)
        assert int(n[0]) == ndoc == 4 + 3 + 4 + 3 + 2 + 2
        kk = len(docs)
        assert kk == 8 and (i[0, kk:] == -1).all()
        assert np.array_equal(s[0, :kk], scores) and np.array_equal(i[0, :kk], docs), (aggr, s[0], i[0], docs, scores)
        if aggr == "add":
            got = dict(zip(i[0, :kk].tolist(), s[0, :kk].tolist()))
            one = np.float32(1 + 2.0 ** -23)
            fold = np.float32(np.float32(np.float32(one + one) + one) + one)
            assert got[0] == fold and got[2] == np.float32(1.5)   # the repeated leaf counts twice
            three = np.float32(np.float32(one + one) + one)
            assert float(three) != 3 * float(one)                 # (the fold does round at c = 3)


@pytest.mark.parametrize("aggr", ["add", "max"])
def test_a_leaf_listing_a_document_twice_counts_twice(aggr):
    """The reference concatenates the leaves' lists, so a document a leaf lists twice is two occurrences (the small64
    golden index has four such leaves).  Document 0 is listed twice in leaf A and once in B; the query asks for B, A."""
    X, Q, _, _ = _exact_case()
    clus = {(0, 0): [0, 0, 2], (0, 1): [0, 5], (1, 1): [0, 6]}
    dec = np.array([[(0, 1), (0, 0)]], np.int64)
    rr = _reranker(X, clus, 4)
    assert rr.index.occurrence_table()[1] == 4
    s, i, n = (t.cpu().numpy() for t in rr.rerank(Q, dec, topk=10, multiclus_score_aggr=aggr))
    (docs, scores, ndoc), = oracle.cluster_rerank(Q, X, clus, dec, multiclus_aggr=aggr)
    assert int(n[0]) == ndoc == 5 and len(docs) == 3 and (i[0, 3:] == -1).all()
    assert np.array_equal(s[0, :3], scores) and np.array_equal(i[0, :3], docs)


def test_negative_scores_aggregate_by_sum_not_by_max():
    """Document 3 (s = -1.5) is listed under two of the query's leaves, document 4 (s = -2) under one.  'add' scores
    document 3 at -3.0, below document 4; 'max' keeps -1.5, above it."""
    X, Q, clus, dec = _exact_case()
    rr = _reranker(X, clus, 4)
    for aggr, want_order in (("add", [4, 3]), ("max", [3, 4])):
        s, i, _ = (t.cpu().numpy() for t in rr.rerank(Q, dec, topk=10, multiclus_score_aggr=aggr))
        ids = i[0].tolist()
        assert [d_ for d_ in ids if d_ in (3, 4)] == want_order
        assert s[0, ids.index(3)] == (np.float32(-3.0) if aggr == "add" else np.float32(-1.5))


@pytest.mark.parametrize("aggr", ["add", "max"])
def test_single_cluster_index_is_unchanged(gauss, aggr):
    from mevi_b200.rerank import ClusterIndex, ClusterReranker

    dec = gauss.load("beam100_labels.npy")
    rr = ClusterReranker(dev(gauss.X), ClusterIndex.from_codes(gauss.codes, gauss.K), mode="stream")
    occ, n_occ = rr.index.occurrence_table()
    assert n_occ == 1 and tuple(occ.shape) == (gauss.n, 0)
    for k in (7, 100):
        s0, i0, n0 = rr.rerank(gauss.Q, dec, topk=k)
        s1, i1, n1 = rr.rerank(gauss.Q, dec, topk=k, multiclus_score_aggr=aggr)
        assert torch.equal(s0, s1) and torch.equal(i0, i1) and torch.equal(n0, n1)


def test_errors(gauss):
    import mevi_b200
    from mevi_b200.rerank import ClusterIndex, ClusterReranker

    dec = gauss.load("beam10_labels.npy")
    rr = ClusterReranker(dev(gauss.X), ClusterIndex.from_codes(gauss.codes, gauss.K), mode="stream")
    with pytest.raises(ValueError, match="'add' or 'max'"):
        rr.rerank(gauss.Q, dec, topk=10, multiclus_score_aggr="sum")
    # a leaf-partitioned shard: its documents' other leaves may live on other ranks
    part = ClusterIndex.from_codes(gauss.codes, gauss.K, doc_ids=torch.arange(gauss.n, dtype=torch.int64))
    with pytest.raises(NotImplementedError):
        ClusterReranker(dev(gauss.X), part, mode="stream").rerank(gauss.Q, dec, topk=10, multiclus_score_aggr="add")
    # a document listed under 17 leaves
    X = np.random.RandomState(0).standard_normal((40, 64)).astype(np.float32)
    clus = {(a, b): [0, 1 + 2 * a + b] for a in range(4) for b in range(4)}
    clus[(4, 0)] = [0]
    rr17 = _reranker(X, clus, 8)
    assert rr17.index.occurrence_table()[1] == 17
    dec17 = np.array([[(a, b) for a in range(4) for b in range(4)]], np.int64)
    with pytest.raises(mevi_b200.MeviError, match="at most 16"):
        rr17.rerank(X[:1], dec17, topk=10, multiclus_score_aggr="max")


def _numpy_occurrence_table(off, docids):
    n = docids.shape[0]
    leaf_of = np.repeat(np.arange(off.shape[0] - 1), np.diff(off))
    order = np.lexsort((np.arange(n), docids))
    groups = np.split(order, np.nonzero(np.diff(docids[order]))[0] + 1) if n else []
    C = max((len(g) for g in groups), default=1)
    occ = np.full((n, C - 1), -1, np.int32)
    for g in groups:
        for p in g:
            others = [(-2 - leaf_of[o] if leaf_of[o] == leaf_of[p] and o < p else leaf_of[o]) for o in g if o != p]
            occ[p, : len(others)] = others
    return occ, C


@pytest.mark.parametrize("which", ["C1", "C2", "C4", "C2-dup"])
def test_occurrence_table_equals_numpy(gauss, which):
    from mevi_b200.rerank import ClusterIndex

    if which == "C1":
        idx = ClusterIndex.from_codes(gauss.codes, gauss.K)
    elif which == "C2":
        idx = ClusterIndex.from_cluster_dict(_golden("gauss768", "multiclus_dict"), gauss.K)
    elif which == "C2-dup":  # small64's index: four leaves list a document twice
        idx = ClusterIndex.from_cluster_dict(_golden("small64", "multiclus_dict"), 16)
    else:
        rs = np.random.RandomState(5)
        clus = {}
        for doc in range(5000):
            for leaf in rs.choice(64, rs.randint(1, 5), replace=False):
                clus.setdefault((int(leaf) // 8, int(leaf) % 8), []).append(doc)
        idx = ClusterIndex.from_cluster_dict(clus, 8)
    occ, C = idx.occurrence_table()
    want, want_C = _numpy_occurrence_table(idx.leaf_offsets.cpu().numpy(), idx.leaf_docids.cpu().numpy())
    assert C == want_C == int(which[1])
    assert np.array_equal(occ.cpu().numpy(), want)
    assert idx.occurrence_table()[0] is occ  # built once per index
