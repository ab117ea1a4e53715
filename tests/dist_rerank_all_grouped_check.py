"""Multi-GPU check of the sharded `rerank_all` on the leaf-grouped scorer (mode="grouped"; NCCL, one process per GPU):
every rank returns the single-GPU streaming answer on the whole index, bit for bit, for row-block shards (single-cluster,
and multi-cluster 'add' / 'max' with C = 2) and for leaf-partitioned shards.
Launch: torchrun --nproc-per-node 2 tests/dist_rerank_all_grouped_check.py"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mevi_b200.dist_utils import shard_bounds  # noqa: E402
from mevi_b200.rerank import ClusterIndex, ClusterReranker, hn_lines_all  # noqa: E402

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
dev = torch.device("cuda", int(os.environ["LOCAL_RANK"]))
rs = np.random.RandomState(0)
n, d, K, nq, L = 30011, 64, 16, 40, 12
X = rs.standard_normal((n, d)).astype(np.float32)
X[n - 500 :] = X[:500]  # exact score ties between documents of the first and the last row block
X[:50, 8:] = 0.0
Q = rs.standard_normal((nq, d)).astype(np.float32)
Q[:, :8] = 0.0  # documents 0..49 score exactly 0
codes = rs.randint(0, K, size=(n, 2)).astype(np.int32)
second = codes.copy()
second[:, 1] = (second[:, 1] + 1 + rs.randint(0, 3, n)) % K
clus = {}
for doc in range(n):  # every document under its own leaf and a neighbouring one (--doc_multiclus 2)
    for c in (codes[doc], second[doc]):
        clus.setdefault((int(c[0]), int(c[1])), []).append(doc)
dec = np.stack([np.stack([rs.choice(K, L, replace=False), rs.choice(K, L)], 1) for _ in range(nq)]).astype(np.int64)
dec[3] = K  # no candidates
texts = [f"query {q}" for q in range(nq)]
Xd = torch.from_numpy(X).to(dev)
s, e = shard_bounds(n, rank, world)

# the single-GPU answers on the whole index, before torch.distributed is initialised
want = {"rows": ClusterReranker(Xd, ClusterIndex.from_codes(codes, K, device_index=dev.index), mode="stream").rerank_all(Q, dec)}
rr_mc = ClusterReranker(Xd, ClusterIndex.from_cluster_dict(clus, K, device_index=dev.index), mode="stream")
assert rr_mc.index.occurrence_table()[1] == 2
for aggr in ("add", "max"):
    want[aggr] = rr_mc.rerank_all(Q, dec, multiclus_score_aggr=aggr)
want["leaf"] = want["rows"]

dist.init_process_group("nccl", device_id=dev)
got = {"rows": ClusterReranker(Xd[s:e], ClusterIndex.from_codes(codes[s:e], K, id_base=s, device_index=dev.index),
                               mode="grouped").rerank_all(Q, dec)}
rr_mc_shard = ClusterReranker(Xd[s:e], ClusterIndex.from_cluster_dict(clus, K, id_base=s, device_index=dev.index, row_range=(s, e)),
                              mode="grouped")
for aggr in ("add", "max"):
    got[aggr] = rr_mc_shard.rerank_all(Q, dec, multiclus_score_aggr=aggr)
    assert rr_mc_shard.last_path == "grouped-all"
index_l, X_own = ClusterIndex.from_sharded_codes(Xd[s:e], torch.from_numpy(codes[s:e]).to(dev), K, s, device_index=dev.index)
rr_l = ClusterReranker(X_own, index_l, mode="grouped")
got["leaf"] = rr_l.rerank_all(Q, dec)
assert rr_l.last_path == "grouped-all"
for tag in ("rows", "add", "max", "leaf"):
    (o1, i1, s1), (o2, i2, s2) = got[tag], want[tag]
    ok = torch.equal(o1, o2) and torch.equal(i1, i2) and torch.equal(s1.view(torch.int32), s2.view(torch.int32))
    lines = hn_lines_all(texts, o1, i1, s1) == hn_lines_all(texts, o2, i2, s2)
    print(f"[grouped rerank_all {tag}] rank {rank}: {int(o2[-1])} candidates, bit-identical {ok}, hn lines equal {lines}", flush=True)
    assert ok and lines, tag
dist.barrier()
if rank == 0:
    print("DIST GROUPED RERANK_ALL CHECK OK", flush=True)
dist.destroy_process_group()
