"""Time the `--doc_multiclus 2` top-k re-rank at full size (8,841,823 x 768, 6,980 queries x 100 leaves).

The corpus is the 4,096-Gaussian mixture of tools/clustered_rerank_time.py.  Every document is listed under its RQ leaf
and, in addition, under the second leaf of its own two-beam `mevi_rq_beam_search`.  Timed, with CUDA events after two
warm-up calls of each:
  (a) rerank(topk=100, multiclus_score_aggr=aggr)            the streaming kernel with the occurrence table
  (b) rerank_all(multiclus_score_aggr=aggr) + truncation     every candidate, aggregated and sorted, then the first 100
  (c) rerank(topk=100) on the single-cluster index            the same corpus, each document under one leaf
  (d) (a) on the leaf-grouped tensor-core path (mode="grouped", the same leaf-ordered matrix plus its fp16 tile image)
(a) is checked against (b), and (d) against (a) bit for bit (ids, fp32 scores, n_candidates); the failed and weak query
counts of (d) are reported.  The working set (27 GB and 54 GB leaf-ordered matrices) is far larger than L2.
Prints one JSON line.  Usage: python tools/multiclus_rerank_time.py [--reps 5] [--queries 6980]"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mevi_b200  # noqa: E402
from mevi_b200.pq import ProductQuantization  # noqa: E402
from mevi_b200.rerank import ClusterIndex, ClusterReranker  # noqa: E402
from mevi_b200.trainer import train_rq_lloyd  # noqa: E402


def leaf_keys(codes, K):
    key = torch.zeros(codes.shape[0], dtype=torch.int64, device=codes.device)
    for j in range(codes.shape[1]):
        key = key * K + codes[:, j].long()
    return key


def multiclus_index(codes, second, K):
    """Inverted lists listing document i under codes[i] and under second[i] (once when they coincide)."""
    n = codes.shape[0]
    k1, k2 = leaf_keys(codes, K), leaf_keys(second, K)
    doc = torch.arange(n, device=codes.device)
    comp = torch.cat([k1 * n + doc, (k2 * n + doc)[k2 != k1]])
    comp, _ = torch.sort(comp)
    keys, counts = torch.unique_consecutive(comp // n, return_counts=True)
    offsets = torch.zeros(keys.numel() + 1, dtype=torch.int64, device=codes.device)
    torch.cumsum(counts, 0, out=offsets[1:])
    return ClusterIndex(keys, offsets, (comp % n).to(torch.int32), codes.shape[1], K)


def timed(fn, reps):
    for _ in range(2):
        out = fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for _ in range(reps):
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    return out, sorted(times)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--queries", type=int, default=6980)
    ap.add_argument("--docs", type=int, default=8841823)
    args = ap.parse_args()
    ctx = mevi_b200.get_context(0)
    dev = torch.device("cuda", 0)
    n, D, K, topk = args.docs, 768, 32, 100
    gc = torch.Generator(device=dev)
    gc.manual_seed(99)
    centers = torch.empty((4096, D), device=dev).normal_(generator=gc)
    gl = torch.Generator(device=dev)
    gl.manual_seed(99 + 1000)
    X = torch.empty((n, D), device=dev)
    for a in range(0, n, 1 << 20):
        b = min(a + (1 << 20), n)
        lab = torch.randint(0, 4096, (b - a,), device=dev, generator=gl)
        X[a:b].normal_(generator=gl).mul_(0.3).add_(centers[lab])
    cb, _ = train_rq_lloyd(X, M=4, K=K, seed=41, iters=10, tol=None, device_index=0, presharded=True)
    codes = ctx.rq_encode(X, cb)
    second = torch.empty_like(codes)
    for a in range(0, n, 1 << 20):
        b = min(a + (1 << 20), n)
        labels, _ = ctx.rq_beam_search(X[a:b].contiguous(), cb, 2)
        second[a:b] = labels[:, 1]
    g = torch.Generator(device=dev)
    g.manual_seed(4321)
    Q = torch.empty((args.queries, D), device=dev).normal_(generator=g)
    pq = ProductQuantization("rq", 4, 5, "l2", D, "kmeans", "grad")
    with torch.no_grad():
        pq.codebook.copy_(cb.cpu())
    dec = torch.cat([pq.beam_search(Q[a:a + 1024], 100) for a in range(0, Q.shape[0], 1024)])

    t0 = time.perf_counter()
    idx_mc = multiclus_index(codes, second, K)
    occ, C = idx_mc.occurrence_table()
    torch.cuda.synchronize()
    build_s = time.perf_counter() - t0
    idx_sc = ClusterIndex.from_codes(codes, K)
    rr_mc = ClusterReranker(None, idx_mc, mode="stream", D_leaf=ctx.gather_rows(X, idx_mc.leaf_docids))
    rr_sc = ClusterReranker(None, idx_sc, mode="stream", D_leaf=ctx.gather_rows(X, idx_sc.leaf_docids))
    del X
    torch.cuda.empty_cache()
    rr_mcg = ClusterReranker(None, idx_mc, mode="grouped", D_leaf=rr_mc.D)  # no third copy: only the fp16 image is added

    def truncated_all(aggr):
        off, ids, scores = rr_mc.rerank_all(Q, dec, multiclus_score_aggr=aggr)
        pos = off[:-1, None] + torch.arange(topk, device=dev)[None, :]
        ok = pos < off[1:, None]
        pos = pos.clamp(max=max(ids.numel() - 1, 0))
        return (torch.where(ok, scores[pos], torch.full_like(scores[pos], float("-inf"))),
                torch.where(ok, ids[pos], torch.full_like(ids[pos], -1)))

    res = dict(n_docs=n, n_positions=int(idx_mc.leaf_docids.numel()), C=int(C), queries=Q.shape[0], leaves=dec.shape[1],
               k=topk, occurrence_table_build_s=round(build_s, 3), gpu=torch.cuda.get_device_name(0))
    try:
        res["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                                            capture_output=True, text=True).stdout.strip()
    except OSError:
        res["power_limit"] = "not read"
    (s_c, i_c, n_c), t_c = timed(lambda: rr_sc.rerank(Q, dec, topk=topk), args.reps)
    res["c_single_cluster_ms"] = t_c
    res["c_mean_candidates"] = float(n_c.float().mean())
    for aggr in ("add", "max"):
        (s_a, i_a, n_a), t_a = timed(lambda: rr_mc.rerank(Q, dec, topk=topk, multiclus_score_aggr=aggr), args.reps)
        (s_b, i_b), t_b = timed(lambda: truncated_all(aggr), args.reps)
        res[f"a_{aggr}_ms"] = t_a
        res[f"b_{aggr}_ms"] = t_b
        res[f"a_{aggr}_mean_candidates"] = float(n_a.float().mean())
        res[f"a_equals_b_{aggr}"] = bool(torch.equal(s_a, s_b) and torch.equal(i_a, i_b))
        (s_d, i_d, n_d), t_d = timed(lambda: rr_mcg.rerank(Q, dec, topk=topk, multiclus_score_aggr=aggr), args.reps)
        res[f"d_{aggr}_ms"] = t_d
        res[f"d_{aggr}_path"] = rr_mcg.last_path
        res[f"d_{aggr}_failed_queries"] = rr_mcg.last_failed_queries
        res[f"d_{aggr}_weak_queries"] = rr_mcg.last_weak_queries
        res[f"d_equals_a_{aggr}"] = bool(torch.equal(i_d, i_a) and torch.equal(s_d.view(torch.int32), s_a.view(torch.int32))
                                         and torch.equal(n_d, n_a))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
