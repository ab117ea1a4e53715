"""Time the sharded `rerank_all` (every candidate of every query, sorted: the shipped recipe's `--save_hard_neg <corpus
size>` output) at full size: 8,841,823 x 768, 6,980 queries, on bench.py's one-GPU corpus (standard normal rows, seed 1234) and
codebook (tests/golden/gauss768/codebook.pt), at L = 10 (marco_eval_nci_rq.sh) and L = 100 leaves per query.

torchrun, one process per GPU; every rank generates the whole corpus with the same seed, keeps its row block
(dist_utils.shard_bounds) and builds its index and leaf-ordered matrix from it.  One call is split into its phases,
each timed with CUDA events after two warm-up calls (medians of --reps calls; the working set is far larger than L2):
  score     mevi_cluster_rerank_all of this rank's candidates (leaf lookup included)
  sort      the segmented sort of them (rerank_all's torch sort)
  exchange  all-gather of the per-rank CSRs (offsets, scores, ids)
  merge     mevi_merge_sorted_runs; its bytes (12 read + 12 written per candidate and pass) over its time against 7.7 TB/s
and the whole `rerank_all` call.  Also: peak device memory per rank over one whole call, and a SHA-256 of the result
(offsets, ids, score bits).  With --ref FILE a world-size-1 run writes its digests there and a larger run compares its
own against them (bit-equality flag).  Prints one JSON line (rank 0).
On one GPU the same run also times, next to the above, the leaf-grouped scorer (mevi_cluster_rerank_all_grouped:
score_grouped_ms, its TFLOP/s from 2 d per candidate against the fp32 FMA bound of 148 SMs x 128 lanes x 2 x 1,965 MHz,
the row bytes each scorer requests), the device sort (mevi_sort_candidates: sort_device_ms, next to the torch sort),
the whole call on each path (rerank_all_stream_ms, rerank_all_grouped_ms), peak extra memory of each whole call
(torch allocations + growth of the library's scratch) and SHA-256 digests of both paths' results, which must agree.
--sweep Q1,Q2,...: also time both scorers at L = 10 on the first Qi queries (the pairs-per-leaf threshold of
mode="auto").
Usage: torchrun --nproc-per-node N tools/dist_rerank_all_time.py [--reps 3] [--leaves 10,100] [--ref FILE] [--out FILE]"""
import argparse
import hashlib
import json
import os
import subprocess
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mevi_b200  # noqa: E402
import mevi_b200.rerank  # noqa: E402
from mevi_b200.dist_utils import all_gather_stack, all_gather_varlen, dist_on, shard_bounds  # noqa: E402
from mevi_b200.pq import ProductQuantization  # noqa: E402
from mevi_b200.rerank import ClusterIndex, ClusterReranker  # noqa: E402

HBM_PEAK = 7.7e12  # bytes/s, B200 data sheet (one GPU)
FP32_FMA_PEAK = 148 * 128 * 2 * 1.965e9  # FLOP/s: 148 SMs x 128 fp32 lanes x 2 x 1,965 MHz boost clock


def digest(off, ids, sc):
    h = hashlib.sha256()
    for t in (off, ids, sc.view(torch.int32)):
        h.update(t.cpu().numpy().tobytes())
    return h.hexdigest()


def median_ms(fn, reps, sync):
    for _ in range(2):
        fn()
    sync()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ts = []
    for _ in range(reps):
        sync()
        a.record()
        fn()
        b.record()
        sync()
        ts.append(a.elapsed_time(b))
    return sorted(ts)[len(ts) // 2]


def extra_memory(fn, sync, dev):
    """(result, GiB): peak device memory of one call above what was allocated before it - torch's allocations plus the
    growth of the library's scratch (cudaMalloc outside torch, seen as free memory lost beyond torch's reserve)."""
    sync()
    torch.cuda.empty_cache()
    free0, res0 = torch.cuda.mem_get_info(dev)[0], torch.cuda.memory_reserved(dev)
    torch.cuda.reset_peak_memory_stats(dev)
    base = torch.cuda.memory_allocated(dev)
    out = fn()
    sync()
    peak = torch.cuda.max_memory_allocated(dev) - base
    torch.cuda.empty_cache()
    lib = max(0, (free0 - torch.cuda.mem_get_info(dev)[0]) - (torch.cuda.memory_reserved(dev) - res0))
    return out, round((peak + lib) / 2**30, 2)


def grouped_times(ctx, rr, index, Q, dec, L, reps, sync, dev):
    """The leaf-grouped scorer and the device sort next to the streaming scorer and the torch sort (one GPU)."""
    d = rr.D.shape[1]
    rg = mevi_b200.rerank.ClusterReranker(None, index, mode="grouped", D_leaf=rr.D)
    ql = index.lookup(dec)
    st = {}
    t = {}
    t["score_grouped_ms"] = median_ms(lambda: st.__setitem__("g", ctx.cluster_rerank_all_grouped(
        Q, rr.D, index.leaf_offsets, index.leaf_docids, ql, id_base=index.id_base)), reps, sync)
    off, sc, ids, _ = st.pop("g")
    out = (torch.empty_like(sc), torch.empty_like(ids))
    t["sort_device_ms"] = median_ms(lambda: ctx.sort_candidates(off, sc, ids, out=out), reps, sync)
    del out, sc, ids
    cand = int(off[-1])
    sizes = index.leaf_offsets[1:] - index.leaf_offsets[:-1]
    valid = ql >= 0
    pairs = torch.bincount(ql[valid].long(), minlength=sizes.numel())
    chunks = (pairs + 255) // 256  # an item meets up to 256 of its leaf's pairs
    t["grouped_tflops"] = round(2 * d * cand / (t["score_grouped_ms"] * 1e-3) / 1e12, 2)
    t["grouped_share_of_fp32_fma_peak"] = round(2 * d * cand / (t["score_grouped_ms"] * 1e-3) / FP32_FMA_PEAK, 3)
    t["row_bytes_stream_gb"] = round(4 * d * cand / 1e9, 1)
    t["row_bytes_grouped_items_gb"] = round(4 * d * int((sizes * chunks).sum()) / 1e9, 1)
    t["row_bytes_distinct_gb"] = round(4 * d * int(sizes[pairs > 0].sum()) / 1e9, 1)
    t["pairs_per_leaf"] = round(ql.numel() / max(1, index.n_leaves), 2)
    t["rerank_all_stream_ms"] = median_ms(lambda: rr.rerank_all(Q, dec), reps, sync)
    t["rerank_all_grouped_ms"] = median_ms(lambda: rg.rerank_all(Q, dec), reps, sync)
    (o1, i1, s1), t["peak_extra_gib_stream"] = extra_memory(lambda: rr.rerank_all(Q, dec), sync, dev)
    d_stream = digest(o1, i1, s1)
    del o1, i1, s1
    (o2, i2, s2), t["peak_extra_gib_grouped"] = extra_memory(lambda: rg.rerank_all(Q, dec), sync, dev)
    t["path_grouped"] = rg.last_path
    d_grouped = digest(o2, i2, s2)
    del o2, i2, s2
    t["digest_stream"], t["digest_grouped"] = d_stream, d_grouped
    t["digests_equal"] = d_stream == d_grouped
    return {k: (round(v, 2) if isinstance(v, float) else v) for k, v in t.items()}


def sweep(ctx, rr, index, Q, dec, counts, reps, sync):
    """Both scorers on the first nq queries: where the grouped one starts to win (mode="auto")."""
    out = []
    for nq in counts:
        q, ql = Q[:nq].contiguous(), index.lookup(dec[:nq])
        a = (q, rr.D, index.leaf_offsets, index.leaf_docids, ql)
        ms_s = median_ms(lambda: ctx.cluster_rerank_all(*a, id_base=index.id_base), reps, sync)
        ms_g = median_ms(lambda: ctx.cluster_rerank_all_grouped(*a, id_base=index.id_base), reps, sync)
        out.append(dict(queries=nq, pairs_per_leaf=round(ql.numel() / max(1, index.n_leaves), 3), score_stream_ms=round(ms_s, 3),
                        score_grouped_ms=round(ms_g, 3)))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--leaves", default="10,100")
    ap.add_argument("--docs", type=int, default=8841823)
    ap.add_argument("--queries", type=int, default=6980)
    ap.add_argument("--ref", default=None)
    ap.add_argument("--sweep", default="")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    local = int(os.environ.get("LOCAL_RANK", 0))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if int(os.environ.get("WORLD_SIZE", 1)) > 1:
        dist.init_process_group("nccl", device_id=dev)
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist_on() else (0, 1)

    def sync():
        torch.cuda.synchronize(dev)
        if dist_on():
            dist.barrier()

    ctx = mevi_b200.get_context(dev.index)
    n, D, K = args.docs, 768, 32
    g = torch.Generator(device=dev)
    g.manual_seed(1234)
    s, e = shard_bounds(n, rank, world)
    Xs = torch.empty((e - s, D), device=dev)
    step = 1 << 20
    for a in range(0, n, step):  # the whole corpus's stream of random numbers, this rank's rows kept
        b = min(a + step, n)
        blk = torch.empty((b - a, D), device=dev).normal_(generator=g)
        lo, hi = max(a, s), min(b, e)
        if lo < hi:
            Xs[lo - s : hi - s] = blk[lo - a : hi - a]
    del blk
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cb_param = torch.load(os.path.join(root, "tests", "golden", "gauss768", "codebook.pt"), map_location="cpu", weights_only=False)
    cb = cb_param.detach().contiguous().to(dev)
    codes = ctx.rq_encode(Xs, cb)
    gq = torch.Generator(device=dev)
    gq.manual_seed(4321)
    Q = torch.empty((args.queries, D), device=dev).normal_(generator=gq)
    pq = ProductQuantization("rq", cb.shape[0], 5, "l2", D, "kmeans", "grad")
    with torch.no_grad():
        pq.codebook.copy_(cb.cpu())
    index = ClusterIndex.from_codes(codes, K, id_base=s, device_index=dev.index)
    rr = ClusterReranker(None, index, mode="stream", D_leaf=ctx.gather_rows(Xs, index.leaf_docids))
    del Xs, codes
    torch.cuda.empty_cache()

    res = dict(world=world, n_docs=n, queries=args.queries, gpu=torch.cuda.get_device_name(dev), reps=args.reps)
    try:
        res["power_limit_clocks"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                                                    "-i", str(dev.index)], capture_output=True, text=True).stdout.strip()
    except OSError:
        res["power_limit_clocks"] = "not read"
    ref = json.load(open(args.ref)) if args.ref and world > 1 and os.path.isfile(args.ref) else None
    digests = {}
    for L in (int(v) for v in args.leaves.split(",")):
        dec = torch.cat([pq.beam_search(Q[a : a + 1024], L) for a in range(0, Q.shape[0], 1024)])
        st = {}

        def score():
            ql = index.lookup(dec)
            st["local"] = ctx.cluster_rerank_all(Q, rr.D, index.leaf_offsets, index.leaf_docids, ql, id_base=s)

        def sort():
            off, sc, ids, _ = st["local"]
            seg = torch.repeat_interleave(torch.arange(Q.shape[0], device=dev), off[1:] - off[:-1])
            order = torch.argsort(ids, stable=True)
            order = order[torch.argsort(sc[order], descending=True, stable=True)]
            order = order[torch.argsort(seg[order], stable=True)]
            st["sorted"] = (off, ids[order], sc[order])

        def exchange():
            off, ids, sc = st["sorted"]
            st["gathered"] = (all_gather_stack(off), all_gather_varlen(sc), all_gather_varlen(ids))

        def merge():
            ro, gs, gi = st["gathered"]
            bases = torch.cumsum(ro[:, -1], 0) - ro[:, -1]
            st["merged"] = ctx.merge_sorted_runs(gs, gi, bases, ro, ro.sum(0))

        t = {"score_ms": median_ms(score, args.reps, sync), "sort_ms": median_ms(sort, args.reps, sync)}
        total = int(st["local"][0][-1])
        if world > 1:
            t["exchange_ms"] = median_ms(exchange, args.reps, sync)
            t["merge_ms"] = median_ms(merge, args.reps, sync)
        else:  # one rank: the exchange is the identity, the merge a copy into the query-major layout (the S = 1 pass)
            st["gathered"] = (st["sorted"][0][None], st["sorted"][2], st["sorted"][1])
            t["merge_ms"] = median_ms(merge, args.reps, sync)
        st.clear()
        t["rerank_all_ms"] = median_ms(lambda: rr.rerank_all(Q, dec), args.reps, sync)
        torch.cuda.reset_peak_memory_stats(dev)
        base_mem = torch.cuda.memory_allocated(dev)
        off, ids, sc = rr.rerank_all(Q, dec)
        sync()
        t["peak_extra_gib_per_rank"] = round((torch.cuda.max_memory_allocated(dev) - base_mem) / 2**30, 2)
        all_total = int(off[-1])
        passes = max(1, (world - 1).bit_length())
        merge_bytes = 24 * all_total * passes
        t["candidates_this_rank"] = total
        t["candidates_all"] = all_total
        t["merge_passes"] = passes
        t["merge_gbps"] = round(merge_bytes / (t["merge_ms"] * 1e-3) / 1e9, 1)
        t["merge_share_of_hbm_peak"] = round(merge_bytes / (t["merge_ms"] * 1e-3) / HBM_PEAK, 3)
        digests[f"L{L}"] = digest(off, ids, sc)
        if ref is not None:
            t["bit_equal_to_n1"] = ref.get(f"L{L}") == digests[f"L{L}"]
        peaks = all_gather_stack(torch.tensor([t["peak_extra_gib_per_rank"]], device=dev)).flatten().tolist()
        t["peak_extra_gib_all_ranks"] = peaks
        del off, ids, sc
        if world == 1:
            t.update(grouped_times(ctx, rr, index, Q, dec, L, args.reps, sync, dev))
        res[f"L{L}"] = {k: (round(v, 2) if isinstance(v, float) else v) for k, v in t.items()}
        del dec
        torch.cuda.empty_cache()
    if world == 1 and args.sweep:
        dec = torch.cat([pq.beam_search(Q[a : a + 1024], 10) for a in range(0, Q.shape[0], 1024)])
        res["auto_sweep_L10"] = sweep(ctx, rr, index, Q, dec, [int(v) for v in args.sweep.split(",")], args.reps, sync)
    if rank == 0 and args.out:
        with open(args.out, "w") as fw:
            json.dump(res, fw, indent=1)
    if rank == 0:
        if args.ref and world == 1:
            with open(args.ref, "w") as fw:
                json.dump(digests, fw)
        print(json.dumps(res), flush=True)
    if dist_on():
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
