"""The multi-cluster top-k (`--doc_multiclus > 1`) on the leaf-grouped tensor-core path (K3g):
`ClusterReranker.rerank(..., multiclus_score_aggr=...)` with a tile image must return what the streaming kernel
(`mevi_cluster_rerank_multiclus`) returns, bit for bit: ids, fp32 scores and n_candidates."""
import numpy as np
import pytest
import torch

from gpu_util import dev
from test_gpu_rerank_multiclus import _golden, _line_scores, _multiplicity, _synthetic

pytestmark = pytest.mark.gpu


def _pair(X, clus, K, **attrs):
    """(stream, grouped) re-rankers over one index and one leaf-ordered matrix; attrs are set on the grouped one."""
    from mevi_b200.rerank import ClusterIndex, ClusterReranker

    idx = ClusterIndex.from_cluster_dict(clus, K)
    st = ClusterReranker(dev(X), idx, mode="stream")
    gr = ClusterReranker(None, idx, mode="grouped", D_leaf=st.D)
    for name, v in attrs.items():
        setattr(gr, name, v)
    return st, gr


def _bit_equal(st, gr, Q, dec, k, aggr, path="grouped-multiclus"):
    s0, i0, n0 = st.rerank(Q, dec, topk=k, multiclus_score_aggr=aggr)
    s1, i1, n1 = gr.rerank(Q, dec, topk=k, multiclus_score_aggr=aggr)
    assert st.last_path == "stream-multiclus"
    if path is not None:
        assert gr.last_path == path, (gr.last_path, gr.last_failed_queries, gr.last_weak_queries)
    bad = torch.nonzero((i0 != i1).any(1)).squeeze(1).tolist()
    assert not bad, f"queries {bad[:5]}: ids differ from the streaming kernel's"
    assert torch.equal(s0.view(torch.int32), s1.view(torch.int32)), "scores are not bit-identical"
    assert torch.equal(n0, n1)
    return s1, i1, n1


# small corpora: a threshold-free bootstrap over the first tiles of 3 leaves, then the rest, so that the sample rounds,
# the compaction and the last round all run
SMALL = dict(PLAN="device", BOOT_LEAVES=3, BOOTSTRAP_MIN=128, PASS_BUDGET=16)


@pytest.mark.parametrize("aggr", ["add", "max"])
@pytest.mark.parametrize("case_name,nb", [("gauss768", 100), ("small64", 10)])
def test_topk_equals_the_executed_reference_loop(case_name, nb, aggr):
    """Against main_models.py:3912-4055 EXECUTED verbatim with doc_multiclus=2, save_hard_neg=200 (the goldens of
    test_gpu_rerank_multiclus), on the grouped path."""
    from conftest import golden_case

    case = golden_case(case_name)
    dec = case.load(f"beam{nb}_labels.npy")
    mc = _golden(case_name, "multiclus_dict")
    fm = _golden(case_name, f"multiclus_{aggr}")
    _, rr = _pair(case.X, mc, case.K)
    s, i, n = (t.cpu().numpy() for t in rr.rerank(case.Q, dec, topk=200, multiclus_score_aggr=aggr))
    assert rr.last_path == "grouped-multiclus" and rr.last_failed_queries == 0
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
def synthetic_pair():
    X, Q, clus, dec, K = _synthetic()
    return (Q, dec) + _pair(X, clus, K, **SMALL)


@pytest.mark.parametrize("plan", ["device", "tiles"])
@pytest.mark.parametrize("aggr", ["add", "max"])
@pytest.mark.parametrize("k", [1, 7, 100, 256])
def test_bit_equal_to_the_streaming_kernel(synthetic_pair, k, aggr, plan):
    Q, dec, st, gr = synthetic_pair
    gr.PLAN = plan
    try:
        _bit_equal(st, gr, Q, dec, k, aggr)
    finally:
        gr.PLAN = "device"
    assert gr.last_failed_queries == 0 and gr.last_weak_queries == 0


def _edge_sets():
    """name -> (X, Q, clus, dec, K): a repeated leaf in the list, a leaf listing a document twice, multiplicities up to
    C = 16, and negative scores with c >= 2."""
    rs = np.random.RandomState(11)
    out = {}
    X, Q, clus, dec, K = _synthetic(seed=1)
    dec = dec.copy()
    dec[1:8, 5] = dec[1:8, 1]      # leaf 1 again at position 5 ...
    dec[1:4, 17] = dec[1:4, 1]     # ... and at 17: c = 3 for its documents
    dec[2, 9] = dec[2, 20]         # a later leaf that also comes earlier
    out["repeated-leaf"] = (X, Q, clus, dec, K)
    X, Q, clus, dec, K = _synthetic(seed=2)
    clus = {leaf: list(docs) for leaf, docs in clus.items()}
    for leaf in list(clus)[::3]:
        docs = clus[leaf]
        docs += [docs[j] for j in rs.choice(len(docs), 5, replace=False)]  # five documents listed twice by this leaf
    out["leaf-lists-twice"] = (X, Q, clus, dec, K)
    # every document under 1..16 distinct leaves (K = 16, M = 2: 256 leaves); a query asks for 40 leaves, so c reaches 16
    n, d = 6000, 64
    X = rs.standard_normal((n, d)).astype(np.float32)
    Q = rs.standard_normal((24, d)).astype(np.float32)
    clus = {}
    hot = rs.choice(256, 40, replace=False)
    for doc in range(n):
        c = 16 if doc < 200 else rs.randint(1, 9)
        leaves = hot[rs.choice(40, c, replace=False)] if doc < 200 else rs.choice(256, c, replace=False)
        for leaf in leaves:
            clus.setdefault((int(leaf) // 16, int(leaf) % 16), []).append(doc)
    dec = np.stack([np.stack([hot // 16, hot % 16], -1)[rs.permutation(40)] for _ in range(24)]).astype(np.int64)
    Q[:12] = X[:12] * np.float32(0.5)  # documents with c = 16 near the top
    out["multiplicity-16"] = (X, Q, clus, dec, 16)
    # all scores negative (documents share a mean direction, queries point away from it); under 'add' a document with c
    # >= 2 ranks far below its single-occurrence score, so a threshold from partial counts would drop true members
    X, Q, clus, dec, K = _synthetic(seed=3)
    m = rs.standard_normal(X.shape[1]).astype(np.float32)
    m /= np.linalg.norm(m)
    X = (X + 12 * m).astype(np.float32)
    Q = (-(np.abs(rs.standard_normal((Q.shape[0], 1))) + 1) * m + 0.1 * Q).astype(np.float32)
    out["negative-scores"] = (X, Q, clus, dec, K)
    return out


EDGES = _edge_sets()


@pytest.mark.parametrize("aggr", ["add", "max"])
@pytest.mark.parametrize("name", list(EDGES))
def test_edge_cases(name, aggr):
    X, Q, clus, dec, K = EDGES[name]
    st, gr = _pair(X, clus, K, **SMALL)
    for k in (10, 100):
        s, i, n = _bit_equal(st, gr, Q, dec, k, aggr)
    C = gr.index.occurrence_table()[1]
    if name == "multiplicity-16":
        assert C == 16
        mult = [_multiplicity(clus, dec[q]) for q in range(len(Q))]
        assert max(max(m_.values()) for m_ in mult) == 16
        assert any(mult[q][int(doc)] == 16 for q in range(12) for doc in i[q, :10].tolist())
    if name == "leaf-lists-twice":
        off, docids = gr.index.leaf_offsets.cpu().numpy(), gr.index.leaf_docids.cpu().numpy()
        assert any(len(set(docids[a:b].tolist())) < b - a for a, b in zip(off[:-1], off[1:]))
    if name == "negative-scores":
        assert (s[:, :k] < 0).all()
        if aggr == "add":  # the kept documents include ones with c >= 2 (their score is the fold, not s)
            ss, ii, _ = st.rerank(Q, dec, topk=k, multiclus_score_aggr="max")
            assert (ss != s).any()


def test_all_queries_weak_are_rerun_by_the_streaming_kernel(synthetic_pair):
    Q, dec, st, gr = synthetic_pair
    gr.BOOTSTRAP_MIN = 10 ** 9
    try:
        for aggr in ("add", "max"):
            _bit_equal(st, gr, Q, dec, 100, aggr, path="grouped-multiclus+stream")
            assert gr.last_weak_queries == len(Q) and gr.last_failed_queries == 0
    finally:
        gr.BOOTSTRAP_MIN = SMALL["BOOTSTRAP_MIN"]


@pytest.mark.parametrize("aggr", ["add", "max"])
def test_reruns_only_the_queries_whose_guarantee_failed(aggr):
    """Near-duplicate documents under one leaf overflow the margin window of the three queries that ask for it."""
    X, Q, clus, dec, K = _synthetic(seed=4)
    nd = 2500
    X[:nd] = X[0] + 1e-6 * np.arange(nd, dtype=np.float32)[:, None]
    clus = {leaf: [doc for doc in docs if doc >= nd] for leaf, docs in clus.items()}
    clus[(0, 0)] = sorted(set(clus.get((0, 0), [])) | set(range(nd)))
    clus[(0, 1)] = sorted(set(clus.get((0, 1), [])) | set(range(0, nd, 2)))  # every other duplicate under a second leaf
    clus = {leaf: docs for leaf, docs in clus.items() if docs}
    dec = dec.copy()
    dec[:3, 0] = (0, 0)
    dec[:3, 1] = (0, 1)
    dec[3:] = np.where((dec[3:, :, :1] == 0) & (dec[3:, :, 1:] <= 1), K, dec[3:])  # the others never see those leaves
    Q[:3] = X[0]
    st, gr = _pair(X, clus, K, **SMALL)
    _bit_equal(st, gr, Q, dec, 100, aggr, path="grouped-multiclus+stream")
    assert 1 <= gr.last_failed_queries <= 3


def boundary_multiclus_set(aggr, k=100, per_query=150, deltas=tuple(2.0 ** -e for e in (24, 22, 20, 17, 14, 10, 6)),
                           seed=5):
    """Documents listed under 1..3 leaves; per query, `per_query` of its candidates with c = 1, 2, 3 (a third each) are
    moved along q so that their aggregated float64 score (c s for 'add', s for 'max') sits at s_k +- delta |q||d|
    (s_k = the query's k-th aggregated float64 score before the move).
    -> (X, Q, clus, dec, K, rel [nq, per_query] achieved, c [nq, per_query])"""
    rs = np.random.RandomState(seed)
    n, d, K, nq, L = 40000, 128, 8, 8, 16  # 64 leaves, a query asks for 16: c = 3 is common
    X = rs.standard_normal((n, d))
    Q = rs.standard_normal((nq, d))
    leaves_of = [rs.choice(64, rs.randint(1, 4), replace=False) for _ in range(n)]
    clus = {}
    for doc, ls in enumerate(leaves_of):
        for leaf in ls:
            clus.setdefault((int(leaf) // K, int(leaf) % K), []).append(doc)
    qleaves = np.stack([rs.choice(64, L, replace=False) for _ in range(nq)])
    dec = np.stack([qleaves // K, qleaves % K], -1).astype(np.int64)
    used = np.zeros(n, bool)
    rel = np.zeros((nq, per_query))
    cs = np.zeros((nq, per_query), np.int64)
    moved = []
    for q in range(nq):
        c = np.array([np.isin(ls, qleaves[q]).sum() for ls in leaves_of])
        cand = np.nonzero(c > 0)[0]
        agg = (X[cand] @ Q[q]) * (c[cand] if aggr == "add" else 1)
        s_k = np.sort(agg)[-k]
        rows = np.concatenate([rs.permutation(np.nonzero((c == cc) & ~used)[0])[: per_query // 3] for cc in (1, 2, 3)])
        assert len(rows) == per_query, "too few candidates with c = 1, 2, 3"
        used[rows] = True
        sgn = np.where(np.arange(per_query) % 2 == 0, 1.0, -1.0)
        dl = np.asarray(deltas)[(np.arange(per_query) // 2) % len(deltas)] * sgn
        cr = c[rows] if aggr == "add" else np.ones(per_query)
        qq = Q[q]
        qn2 = qq @ qq
        x = X[rows]
        for _ in range(2):  # |d| moves with d
            target = (s_k + dl * np.sqrt(qn2) * np.linalg.norm(x, axis=1)) / cr
            x = x + ((target - x @ qq) / qn2)[:, None] * qq[None]
        X[rows] = x
        moved.append((rows, s_k, cr))
        cs[q] = c[rows]
    X = X.astype(np.float32)
    Q = Q.astype(np.float32)
    X64, Q64 = X.astype(np.float64), Q.astype(np.float64)
    for q, (rows, s_k, cr) in enumerate(moved):
        rel[q] = (cr * (X64[rows] @ Q64[q]) - s_k) / (np.linalg.norm(Q64[q]) * np.linalg.norm(X64[rows], axis=1))
    for cc in (1, 2, 3):  # the boundary is covered: both sides, within 2^-20, for every c
        r = rel[cs == cc]
        assert (np.abs(r) <= 2.0 ** -20).sum() >= 4 and (r > 0).any() and (r < 0).any(), cc
    assert (np.abs(rel) <= 2.0 ** -5).all()
    return X, Q, clus, dec, K, rel, cs


@pytest.mark.parametrize("aggr", ["add", "max"])
def test_boundary_documents(aggr):
    """Aggregated scores on the boundary: no true member lost, every score bit-equal to the streaming kernel's."""
    X, Q, clus, dec, K, _, _ = boundary_multiclus_set(aggr)
    st, gr = _pair(X, clus, K, PLAN="device", BOOT_LEAVES=(2, 8))
    s0, i0, _ = st.rerank(Q, dec, topk=100, multiclus_score_aggr=aggr)
    s1, i1, _ = gr.rerank(Q, dec, topk=100, multiclus_score_aggr=aggr)
    lost = sum(len(set(i0[q].tolist()) - set(i1[q].tolist())) for q in range(len(Q)))
    assert gr.last_path == "grouped-multiclus" and lost == 0, (gr.last_path, lost)
    assert torch.equal(i0, i1) and torch.equal(s0.view(torch.int32), s1.view(torch.int32))


def test_adversarial_rounding_with_four_occurrences():
    """fp16 rounding errors near the bound, pointing the wrong way (adversarial_rounding_docs), with every document
    listed under the four leaves the query asks for: under 'add' the errors add up four times, so the weakest true
    members are found only through a margin that grows with c."""
    from test_gpu_prefilter_bounds import adversarial_rounding_docs

    D, q, members = adversarial_rounding_docs()
    k = len(members)
    # 40 groups of 500 documents; group g is listed by the leaves (g, 0) .. (g, 3), and the query asks for all 160 leaves,
    # the (g, 0) first: the threshold samples (first tiles of the leading leaves) then hold distinct documents
    G = 40
    groups = np.array_split(np.arange(D.shape[0]), G)
    clus = {(g, j): groups[g].tolist() for g in range(G) for j in range(4)}
    dec = np.array([[(g, j) for j in range(4) for g in range(G)]], np.int64)
    st, gr = _pair(D, clus, 64, BOOTSTRAP_MIN=0)  # no query is weak: thresholds from the grouped rounds only
    for aggr in ("add", "max"):
        s, i, _ = _bit_equal(st, gr, q, dec, k, aggr)
        assert set(i[0].tolist()) == set(members.tolist()), f"{aggr}: {len(set(members) - set(i[0].tolist()))} members missing"


@pytest.mark.parametrize("aggr", ["add", "max"])
def test_single_cluster_index(gauss, aggr):
    """C = 1 (empty occurrence table): bit-equal to the streaming kernel, and the plain grouped rerank() up to the order
    of equal scores."""
    from mevi_b200.rerank import ClusterIndex, ClusterReranker

    dec = gauss.load("beam100_labels.npy")
    idx = ClusterIndex.from_codes(gauss.codes, gauss.K)
    st = ClusterReranker(dev(gauss.X), idx, mode="stream")
    gr = ClusterReranker(None, idx, mode="grouped", D_leaf=st.D)
    assert idx.occurrence_table()[1] == 1
    for k in (7, 100):
        s, i, n = _bit_equal(st, gr, gauss.Q, dec, k, aggr)
        s2, i2, n2 = gr.rerank(gauss.Q, dec, topk=k)
        assert gr.last_path == "grouped" and torch.equal(n, n2)
        assert torch.equal(s.view(torch.int32), s2.view(torch.int32))
        for q in range(len(gauss.Q)):
            a = sorted(zip((-s[q]).tolist(), i[q].tolist()))
            b = sorted(zip((-s2[q]).tolist(), i2[q].tolist()))
            assert a == b


def test_auto_mode():
    """mode='auto' on a corpus of AUTO_MIN_DOCS rows: the grouped path when the queries share leaves, the streaming
    kernel when (query, leaf) pairs per leaf are fewer than AUTO_QUERIES_PER_LEAF."""
    from mevi_b200.rerank import ClusterIndex, ClusterReranker

    X, Q, clus, dec, K = _synthetic(nq=64, n=140000, L=16, seed=6)
    idx = ClusterIndex.from_cluster_dict(clus, K)
    st = ClusterReranker(dev(X), idx, mode="stream")
    auto = ClusterReranker(None, idx, mode="auto", D_leaf=st.D)
    assert st.D.shape[0] >= auto.AUTO_MIN_DOCS and auto._grouped is not None
    assert dec.shape[0] * dec.shape[1] >= auto.AUTO_QUERIES_PER_LEAF * idx.n_leaves
    for aggr in ("add", "max"):
        _bit_equal(st, auto, Q, dec, 100, aggr, path="grouped-multiclus")
        _bit_equal(st, auto, Q[:8], dec[:8], 100, aggr, path="stream-multiclus")
