"""world_size-2 (gloo, CPU) coverage of the sequencing of a sharded `ClusterReranker.rerank_all`: the local scoring and
sort on every rank, the all-gather of the per-rank CSRs and the merge of the sorted runs, on row-block shards (single-
and multi-cluster) and on leaf-partitioned shards.  The two kernel calls are replaced by numpy test doubles (scores as
fp32 roundings of float64 dots, so a candidate scores the same on whichever rank owns it; the merge as a lexsort);
what is under test is mevi_b200/rerank.py and dist_utils.py."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N, D, K, NQ, L = 601, 16, 4, 9, 5


class _Ctx:
    """numpy stand-ins for Context.cluster_rerank_all and Context.merge_sorted_runs."""

    def cluster_rerank_all(self, Q, D_leaf, leaf_offsets, leaf_docids, query_leaves, id_base=0):
        off, ld, ql = leaf_offsets.numpy(), leaf_docids.numpy(), query_leaves.numpy()
        Q64, D64 = Q.numpy().astype(np.float64), D_leaf.numpy().astype(np.float64)
        offsets, scores, ids = [0], [], []
        for q in range(ql.shape[0]):
            rows = np.concatenate([np.arange(off[l], off[l + 1]) for l in ql[q] if l >= 0] + [np.zeros(0, np.int64)])
            scores.append((D64[rows] @ Q64[q]).astype(np.float32))
            ids.append(ld[rows].astype(np.int64) + id_base)
            offsets.append(offsets[-1] + rows.size)
        offsets = torch.tensor(offsets, dtype=torch.int64)
        ncand = (offsets[1:] - offsets[:-1]).to(torch.int32)
        return offsets, torch.from_numpy(np.concatenate(scores)), torch.from_numpy(np.concatenate(ids)), ncand

    def merge_sorted_runs(self, scores_in, ids_in, bases, run_offsets, out_offsets):
        s, i, b, ro = scores_in.numpy(), ids_in.numpy(), bases.numpy(), run_offsets.numpy()
        out_s, out_i = [], []
        for q in range(ro.shape[1] - 1):
            seg = np.concatenate([np.arange(b[r] + ro[r, q], b[r] + ro[r, q + 1]) for r in range(ro.shape[0])])
            order = np.lexsort((i[seg], -s[seg]))
            out_s.append(s[seg][order])
            out_i.append(i[seg][order])
        assert int(out_offsets[-1]) == sum(x.size for x in out_s)
        return torch.from_numpy(np.concatenate(out_s)), torch.from_numpy(np.concatenate(out_i))


class _Index:
    """The fields of ClusterIndex that rerank_all reads, over rows (local row i = document doc_of_row[i])."""

    def __init__(self, leaves_of_row, rows, id_base=0, doc_ids=None):
        pairs = sorted((leaf, r) for r in rows for leaf in leaves_of_row[r])
        self.keys = sorted({leaf for leaf, _ in pairs})
        counts = [sum(1 for leaf, _ in pairs if leaf == k) for k in self.keys]
        self.leaf_offsets = torch.tensor(np.concatenate([[0], np.cumsum(counts)]), dtype=torch.int64)
        self.leaf_docids = torch.tensor([r - rows[0] if doc_ids is None else rows.index(r) for _, r in pairs], dtype=torch.int32)
        self.id_base, self.doc_ids = id_base, doc_ids

    def lookup(self, dec):
        pos = {k: i for i, k in enumerate(self.keys)}
        return torch.tensor([[pos.get(int(l), -1) for l in row] for row in dec], dtype=torch.int32)


def _data():
    rs = np.random.RandomState(7)
    X = rs.standard_normal((N, D)).astype(np.float32)
    X[N - 40 :] = X[:40]  # exact score ties between documents that the row blocks put on different ranks
    Q = rs.standard_normal((NQ, D)).astype(np.float32)
    first = rs.randint(0, K * K, N)
    second = (first + 1 + rs.randint(0, 3, N)) % (K * K)
    dec = np.stack([rs.choice(K * K, L, replace=False) for _ in range(NQ)])
    dec[0] = K * K  # a query without candidates
    dec[1, 1] = dec[1, 0]  # a leaf repeated in a query's list
    return X, Q, first, second, dec


def _reranker(X, rows, leaves_of_row, id_base=0, doc_ids=None):
    from mevi_b200.rerank import ClusterReranker

    rr = ClusterReranker.__new__(ClusterReranker)
    rr.ctx, rr.leaf_ordered = _Ctx(), True
    rr.index = _Index(leaves_of_row, rows, id_base, doc_ids)
    rr.D = torch.from_numpy(X[rows][rr.index.leaf_docids.numpy()])
    return rr


def _cases(first, second):
    single = [(int(a),) for a in first]
    multi = [(int(a), int(b)) for a, b in zip(first, second)]
    return single, multi


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(1)
    from mevi_b200.dist_utils import shard_bounds

    X, Q, first, second, dec = _data()
    single, multi = _cases(first, second)
    s, e = shard_bounds(N, rank, world)
    res = {}
    res["rows"] = _reranker(X, list(range(s, e)), single, id_base=s).rerank_all(Q, dec)
    for aggr in ("add", "max"):
        res[aggr] = _reranker(X, list(range(s, e)), multi, id_base=s).rerank_all(Q, dec, multiclus_score_aggr=aggr)
    # leaf-partitioned: leaves with key % world == rank live here, their rows in an arbitrary order, ids by doc_ids
    own = [r for r in range(N) if first[r] % world == rank][::-1]
    part = _reranker(X, own, single, doc_ids=torch.tensor(own, dtype=torch.int64))
    res["leaf"] = part.rerank_all(Q, dec)
    part_mc = _reranker(X, own, multi, doc_ids=torch.tensor(own, dtype=torch.int64))
    with pytest.raises(NotImplementedError):
        part_mc.rerank_all(Q, dec, multiclus_score_aggr="add")
    for name, (off, ids, sc) in res.items():
        np.savez(os.path.join(out_dir, f"{name}_{rank}.npz"), off=off.numpy(), ids=ids.numpy(), sc=sc.numpy())
    dist.barrier()  # no rank hangs after the refused call
    dist.destroy_process_group()


def test_sharded_rerank_all_equals_single_rank(tmp_path):
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    world = 2
    mp.spawn(_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    X, Q, first, second, dec = _data()
    single, multi = _cases(first, second)
    rows = list(range(N))
    want = {"rows": _reranker(X, rows, single).rerank_all(Q, dec), "leaf": _reranker(X, rows, single).rerank_all(Q, dec)}
    for aggr in ("add", "max"):
        want[aggr] = _reranker(X, rows, multi).rerank_all(Q, dec, multiclus_score_aggr=aggr)
    assert int(want["rows"][0][1]) == 0 and int(want["rows"][0][-1]) > 0
    for name, (off, ids, sc) in want.items():
        for rank in range(world):
            got = np.load(tmp_path / f"{name}_{rank}.npz")
            assert np.array_equal(got["off"], off.numpy()), (name, rank)
            assert np.array_equal(got["ids"], ids.numpy()), (name, rank)
            assert np.array_equal(got["sc"].view(np.int32), sc.numpy().view(np.int32)), (name, rank)


def test_leaf_partitioned_rerank_all_without_distributed_maps_rows_to_documents():
    """A doc_ids index outside torch.distributed: the same answer as the plain index, ties ordered by document id."""
    X, Q, first, second, dec = _data()
    single, multi = _cases(first, second)
    rows = list(range(N))
    perm = list(np.random.RandomState(1).permutation(N))
    off, ids, sc = _reranker(X, rows, single).rerank_all(Q, dec)
    off2, ids2, sc2 = _reranker(X, perm, single, doc_ids=torch.tensor(perm, dtype=torch.int64)).rerank_all(Q, dec)
    assert torch.equal(off, off2) and torch.equal(ids, ids2) and torch.equal(sc.view(torch.int32), sc2.view(torch.int32))
    with pytest.raises(NotImplementedError):
        _reranker(X, perm, multi, doc_ids=torch.tensor(perm, dtype=torch.int64)).rerank_all(Q, dec, multiclus_score_aggr="max")
