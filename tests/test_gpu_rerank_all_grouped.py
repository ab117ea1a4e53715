"""The leaf-grouped every-candidate scorer and the device candidate sort behind `ClusterReranker.rerank_all`:
mevi_cluster_rerank_all_grouped equals mevi_cluster_rerank_all byte for byte (score bits, ids, n_candidates);
mevi_sort_candidates equals the three stable torch passes bit for bit; rerank_all's "grouped" and "auto" modes equal
"stream"; and a sharded grouped call on two GPUs equals the one-GPU call (tests/dist_rerank_all_grouped_check.py)."""
import math
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from gpu_util import ctx, dev

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _same_scores(a, b):
    (oa, sa, ia, na), (ob, sb, ib, nb) = a, b
    assert torch.equal(oa, ob)
    assert torch.equal(sa.view(torch.int32), sb.view(torch.int32)), "score bits differ"
    assert torch.equal(ia, ib)
    assert torch.equal(na, nb)


def _both(X, Q, sizes, ql, id_base=0):
    """Both scorers on a raw leaf-ordered index (leaves of the given sizes, rows in leaf order, shuffled ids)."""
    c = ctx()
    sizes = np.asarray(sizes, np.int64)
    off = dev(np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64))
    ld = dev(np.random.RandomState(5).permutation(X.shape[0]).astype(np.int32))
    args = (dev(Q), dev(X), off, ld, dev(np.ascontiguousarray(ql, dtype=np.int32)))
    a = c.cluster_rerank_all(*args, id_base=id_base)
    b = c.cluster_rerank_all_grouped(*args, id_base=id_base)
    return a, b


SIZES = [1, 127, 128, 129, 0, 300, 513, 2, 64]


def _ql(rs, nq, L, n_leaves):
    ql = rs.randint(-1, n_leaves, size=(nq, L)).astype(np.int32)
    ql[:, 0] = 5       # one leaf chosen by every query: more than a pass (32) and an item (256) of pairs
    ql[:, 1] = 5       # ... and repeated in every query's list
    ql[0, :] = -1      # a query without candidates
    if nq > 2:
        ql[1, :] = 4   # only an empty leaf
    return ql


@pytest.mark.parametrize("d", [4, 64, 196, 768, 1024])
def test_grouped_scorer_equals_streaming_bytes(d):
    rs = np.random.RandomState(d)
    n = sum(SIZES)
    X = rs.standard_normal((n, d)).astype(np.float32)
    Q = rs.standard_normal((150, d)).astype(np.float32)
    a, b = _both(X, Q, SIZES, _ql(rs, 150, 7, len(SIZES)), id_base=1000)
    assert int(a[0][-1]) > 256 * 128
    _same_scores(a, b)


def test_grouped_scorer_single_query_and_every_leaf():
    rs = np.random.RandomState(1)
    n = sum(SIZES)
    X = rs.standard_normal((n, 768)).astype(np.float32)
    Q = rs.standard_normal((1, 768)).astype(np.float32)
    ql = np.array([[3, -1, 0, 1, 2, 4, 5, 6, 7, 8, 3, -1]], np.int32)  # a repeat, -1 and an empty leaf
    _same_scores(*_both(X, Q, SIZES, ql))


@pytest.mark.parametrize("scale", [1.0, 2.0 ** -30, 2.0 ** 20])
@pytest.mark.parametrize("d", [64, 768])
def test_grouped_scorer_zeros_signed_zeros_and_scales(d, scale):
    """Zero and negative-zero rows and queries, rows that are zero in half their columns: zero lane partials and the
    sign of a zero score; inputs scaled far down and up."""
    rs = np.random.RandomState(7)
    n = sum(SIZES)
    X = (rs.standard_normal((n, d)) * scale).astype(np.float32)
    Q = (rs.standard_normal((40, d)) * scale).astype(np.float32)
    X[::7] = 0.0
    X[1::7] = -0.0
    X[2::7, : d // 2] = -0.0
    X[3::7, d // 2 :] = 0.0
    X[4::7] = -X[4::7]
    Q[2] = -0.0
    Q[3] = 0.0
    Q[4, ::2] = -0.0
    a, b = _both(X, Q, SIZES, _ql(rs, 40, 6, len(SIZES)))
    assert int((a[1].view(torch.int32) == 0).sum()) > 0  # +0.0 scores (zero rows and queries)
    _same_scores(a, b)


@pytest.mark.parametrize("nb", [10, 100])
def test_grouped_scorer_on_golden_cases(case, nb):
    from mevi_b200.rerank import ClusterIndex

    c = ctx()
    idx = ClusterIndex.from_codes(case.codes, case.K)
    D = c.gather_rows(dev(case.X), idx.leaf_docids)
    ql = idx.lookup(case.load(f"beam{nb}_labels.npy"))
    Q = dev(case.Q)
    _same_scores(c.cluster_rerank_all(Q, D, idx.leaf_offsets, idx.leaf_docids, ql),
                 c.cluster_rerank_all_grouped(Q, D, idx.leaf_offsets, idx.leaf_docids, ql))


# ---- the candidate sort ----------------------------------------------------------------------------------------------
def _torch_sorted(off, s, i):
    from mevi_b200.rerank import sort_candidates_torch

    return sort_candidates_torch(off, s, i)


def _check_sort(counts, scores, ids):
    c = ctx()
    counts = np.asarray(counts, np.int64)
    off = dev(np.concatenate([[0], np.cumsum(counts)]).astype(np.int64))
    s, i = dev(np.asarray(scores, np.float32)), dev(np.asarray(ids, np.int64))
    ws, wi = _torch_sorted(off, s, i)
    gs, gi = c.sort_candidates(off, s, i)
    assert torch.equal(gi, wi)
    assert torch.equal(gs.view(torch.int32), ws.view(torch.int32))
    s2, i2 = s.clone(), i.clone()  # in place
    c.sort_candidates(off, s2, i2, out=(s2, i2))
    assert torch.equal(i2, wi) and torch.equal(s2.view(torch.int32), ws.view(torch.int32))


@pytest.mark.parametrize("total", [100, 4096, 4097, 1 << 17, 3_000_000])
def test_sort_equals_torch_passes_with_ties(total):
    rs = np.random.RandomState(total % 1000)
    nq = max(1, total // 700)
    cuts = np.sort(rs.randint(0, total + 1, nq - 1))
    counts = np.diff(np.concatenate([[0], cuts, [total]]))
    scores = (rs.randint(-6, 7, total) / 4.0).astype(np.float32)  # many exact ties
    ids = rs.randint(0, 5000, total)                                 # ... also in (score, id)
    _check_sort(counts, scores, ids)


@pytest.mark.parametrize("total", [64, 5000, 1 << 16])
def test_sort_special_values(total):
    rs = np.random.RandomState(3)
    special = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 1e-40, -1e-40, 1e-45, -1e-45, 3.0, -3.0], np.float32)
    scores = special[rs.randint(0, len(special), total)]
    ids = rs.randint(0, 50, total)
    counts = [0, total // 3, 0, total - total // 3, 0]
    _check_sort(counts, scores, ids)


def test_sort_one_segment_empty_segments_and_nothing():
    rs = np.random.RandomState(4)
    scores = rs.standard_normal(20000).astype(np.float32)
    _check_sort([20000], scores, rs.permutation(20000))
    _check_sort([0, 0, 20000, 0], scores, rs.permutation(20000))
    _check_sort([0, 0, 0], np.zeros(0, np.float32), np.zeros(0, np.int64))


def test_sort_id_range():
    from mevi_b200._lib import MeviError

    top = (1 << 32) - 1
    _check_sort([3], [1.0, 1.0, 2.0], [top, 0, top - 5])
    c = ctx()
    off = dev(np.array([0, 3], np.int64))
    for bad in (1 << 32, -1):
        with pytest.raises(MeviError, match="2\\^32"):
            c.sort_candidates(off, dev(np.ones(3, np.float32)), dev(np.array([0, bad, 2], np.int64)))


def test_sort_above_two_to_the_31_elements():
    """Two queries of 2^30 + 2,049 and 2^30 + 2,050 candidates (ids 0..m-1, score = (id * 7919) % 1024: every score ties
    with about a million others): each output segment is ordered by (score desc, id asc), holds every id once, and
    keeps every id's score.  Skipped without about 100 GB of free device memory."""
    free = torch.cuda.mem_get_info(0)[0]
    if free < 100 * (1 << 30):
        pytest.skip("needs ~100 GB of free device memory")
    c = ctx()
    m = [(1 << 30) + 2049, (1 << 30) + 2050]
    off = torch.tensor([0, m[0], m[0] + m[1]], dtype=torch.int64, device="cuda:0")
    ids = torch.cat([torch.arange(k, dtype=torch.int64, device="cuda:0").flip(0) for k in m])
    scores = ((ids * 7919) % 1024).to(torch.float32)
    c.sort_candidates(off, scores, ids, out=(scores, ids))
    step = 1 << 27
    for q in range(2):
        a, b = int(off[q]), int(off[q + 1])
        seen = torch.zeros(m[q], dtype=torch.bool, device="cuda:0")
        seen[ids[a:b]] = True
        assert bool(seen.all())
        del seen
        for lo in range(a, b - 1, step):
            hi = min(lo + step + 1, b)
            s, i = scores[lo:hi], ids[lo:hi]
            assert torch.equal(s, ((i * 7919) % 1024).to(torch.float32))
            ok = (s[:-1] > s[1:]) | ((s[:-1] == s[1:]) & (i[:-1] < i[1:]))
            assert bool(ok.all())


# ---- rerank_all ------------------------------------------------------------------------------------------------------
def _equal_csr(a, b):
    (o1, i1, s1), (o2, i2, s2) = a, b
    assert torch.equal(o1, o2) and torch.equal(i1, i2) and torch.equal(s1.view(torch.int32), s2.view(torch.int32))


@pytest.mark.parametrize("nb", [10, 100])
def test_rerank_all_modes_equal_on_golden_cases(case, nb):
    from mevi_b200.rerank import ClusterIndex, ClusterReranker, sort_candidates_torch

    dec = case.load(f"beam{nb}_labels.npy")
    idx = ClusterIndex.from_codes(case.codes, case.K)
    rs = ClusterReranker(dev(case.X), idx, mode="stream")
    want = rs.rerank_all(case.Q, dec)
    assert rs.last_path == "stream-all"
    rg = ClusterReranker(None, idx, mode="grouped", D_leaf=rs.D)
    _equal_csr(rg.rerank_all(case.Q, dec), want)
    assert rg.last_path == "grouped-all"
    ra = ClusterReranker(None, idx, mode="auto", D_leaf=rs.D)
    _equal_csr(ra.rerank_all(case.Q, dec), want)
    # the torch restatement of the sort on the unsorted scores
    off, sc, ids, _ = ctx().cluster_rerank_all(dev(case.Q), rs.D, idx.leaf_offsets, idx.leaf_docids, idx.lookup(dec))
    ws, wi = sort_candidates_torch(off, sc, ids)
    _equal_csr((off, wi, ws), want)


@pytest.mark.parametrize("aggr", ["add", "max"])
def test_rerank_all_modes_equal_multiclus(gauss, aggr):
    from mevi_b200.rerank import ClusterIndex, ClusterReranker

    dec = gauss.load("beam100_labels.npy")
    clus = {k: list(v) for k, v in gauss.pickle("rqclus.pkl").items()}
    keys = sorted(clus)
    for j, k in enumerate(keys):  # every document of a leaf also listed under the next leaf
        clus[keys[(j + 1) % len(keys)]] = sorted(set(clus[keys[(j + 1) % len(keys)]]) | set(clus[k][:5]))
    idx = ClusterIndex.from_cluster_dict(clus, gauss.K)
    assert idx.occurrence_table()[1] >= 2
    rs = ClusterReranker(dev(gauss.X), idx, mode="stream")
    want = rs.rerank_all(gauss.Q, dec, multiclus_score_aggr=aggr)
    rg = ClusterReranker(None, idx, mode="grouped", D_leaf=rs.D)
    _equal_csr(rg.rerank_all(gauss.Q, dec, multiclus_score_aggr=aggr), want)
    assert rg.last_path == "grouped-all"


def test_rerank_all_modes_equal_on_a_doc_ids_index(gauss):
    from mevi_b200.rerank import ClusterIndex, ClusterReranker

    dec = gauss.load("beam100_labels.npy")
    perm = np.random.RandomState(3).permutation(gauss.n)
    part = ClusterIndex.from_codes(gauss.codes[perm], gauss.K, doc_ids=torch.from_numpy(perm))
    X = dev(gauss.X[perm])
    want = ClusterReranker(X, part, mode="stream").rerank_all(gauss.Q, dec)
    got = ClusterReranker(X, part, mode="grouped").rerank_all(gauss.Q, dec)
    _equal_csr(got, want)
    plain = ClusterReranker(dev(gauss.X), ClusterIndex.from_codes(gauss.codes, gauss.K), mode="grouped").rerank_all(gauss.Q, dec)
    _equal_csr(plain, want)


def test_rerank_all_auto_selection(gauss):
    from mevi_b200.rerank import ClusterIndex, ClusterReranker

    dec = gauss.load("beam100_labels.npy")
    idx = ClusterIndex.from_codes(gauss.codes, gauss.K)
    rr = ClusterReranker(dev(gauss.X), idx, mode="auto")
    need = ClusterReranker.AUTO_ALL_QUERIES_PER_LEAF * idx.n_leaves
    many = math.ceil(need / dec.shape[1])  # fewest queries that reach the threshold
    assert many <= dec.shape[0]
    want = ClusterReranker(None, idx, mode="stream", D_leaf=rr.D).rerank_all(gauss.Q[:many], dec[:many])
    _equal_csr(rr.rerank_all(gauss.Q[:many], dec[:many]), want)
    assert rr.last_path == "grouped-all"
    few = many - 1
    if few >= 1:
        rr.rerank_all(gauss.Q[:few], dec[:few])
        assert rr.last_path == "stream-all"


def test_sharded_grouped_rerank_all_on_two_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "dist_rerank_all_grouped_check.py")],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0 and "DIST GROUPED RERANK_ALL CHECK OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
