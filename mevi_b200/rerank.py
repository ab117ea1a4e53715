"""Cluster-restricted re-rank: the loop of MEVI/main_models.py:3911-4053 as one kernel launch.

The reference walks, per query, the RQ leaves emitted by NCI beam search,
looks each leaf up in the `rqclus` dictionary (3928), fancy-indexes the
candidate rows out of the doc-embedding memmap (3944 / IndexedData 1011-1017),
copies them to the GPU in chunks of `encode_batch_size` (3948-3952), scores
q.P^T (3967-3968), concatenates and sorts (4012-4014), then prints the hn /
fine lines (4046-4053, 4082).  Here the inverted lists live on the device as
CSR, all queries go through `mevi_cluster_rerank` at once, and only the k best
come back.  Text output keeps the reference's byte format.
"""
from __future__ import annotations

import pickle
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from .dist_utils import all_gather_stack, all_gather_varlen, dist_on, rank_world, shard_bounds


class ClusterIndex:
    """Inverted lists leaf -> doc ids on the device (CSR over the non-empty leaves).

    leaf_keys    int64 [n_leaves]   sorted base-K value of the code tuple
    leaf_offsets int64 [n_leaves+1]
    leaf_docids  int32 [n]          local row indices, ascending inside a leaf
    """

    def __init__(self, leaf_keys, leaf_offsets, leaf_docids, M: int, K: int, id_base: int = 0, doc_ids=None):
        self.leaf_keys, self.leaf_offsets, self.leaf_docids = leaf_keys, leaf_offsets, leaf_docids
        self.M, self.K, self.id_base = int(M), int(K), int(id_base)
        # int64 [n] or None: document id of local row i when the rows are not one contiguous id range (a leaf-partitioned
        # shard, dist_utils.partition_rows_by_leaf); results are then doc_ids[row] instead of id_base + row
        self.doc_ids = doc_ids
        self._occ = None

    @property
    def n_leaves(self) -> int:
        return int(self.leaf_keys.numel())

    @property
    def device(self):
        return self.leaf_keys.device

    # -- construction -------------------------------------------------------
    @classmethod
    def from_codes(cls, codes, K: int, id_base: int = 0, device_index: Optional[int] = None, doc_ids=None) -> "ClusterIndex":
        """Replaces the dict loops of pq.py:236-242 / 200-214 with a device sort by leaf key."""
        ctx = _lib.get_context(device_index)
        dev = torch.device("cuda", ctx.device)
        if not isinstance(codes, torch.Tensor):
            codes = torch.from_numpy(np.ascontiguousarray(codes, dtype=np.int32))
        codes = codes.to(device=dev, dtype=torch.int32).contiguous()
        M = codes.shape[1]
        docids, keys = ctx.build_inverted_lists(codes, K)
        leaf_keys, counts = torch.unique_consecutive(keys, return_counts=True)
        offsets = torch.zeros(leaf_keys.numel() + 1, dtype=torch.int64, device=dev)
        torch.cumsum(counts, 0, out=offsets[1:])
        if doc_ids is not None:
            assert id_base == 0 and doc_ids.numel() == codes.shape[0]
            doc_ids = doc_ids.to(device=dev, dtype=torch.int64).contiguous()
        return cls(leaf_keys, offsets, docids, M, K, id_base, doc_ids)

    @classmethod
    def from_sharded_codes(cls, X_local, codes_local, K: int, id_base: int, device_index: Optional[int] = None):
        """Leaf-partitioned index of a row-block-sharded corpus (torch.distributed initialised): every leaf is moved,
        whole, to one rank (`dist_utils.partition_rows_by_leaf`).  -> (index, X_own): this rank's leaves and their rows."""
        from .dist_utils import partition_rows_by_leaf

        ctx = _lib.get_context(device_index)
        X_own, codes_own, gids = partition_rows_by_leaf(X_local, codes_local.to(torch.int32), K, id_base, gather_rows=ctx.gather_rows)
        return cls.from_codes(codes_own, K, device_index=device_index, doc_ids=gids), X_own

    @classmethod
    def from_cluster_dict(cls, doc_cluster: Dict[Tuple[int, ...], Sequence[int]], K: int, id_base: int = 0,
                          device_index: Optional[int] = None, row_range: Optional[Tuple[int, int]] = None) -> "ClusterIndex":
        """Load a reference-format `rqclus*.pkl` dictionary (main_models.py:3214-3219).  With
        `row_range=(start, end)` only doc ids of that row block are kept (doc-sharded re-rank)."""
        ctx = _lib.get_context(device_index)
        dev = torch.device("cuda", ctx.device)
        M = len(next(iter(doc_cluster))) if doc_cluster else 1
        keys, lens, ids = [], [], []
        for t, docs in doc_cluster.items():
            key = 0
            for c in t:
                key = key * K + int(c)
            d = np.asarray(docs, dtype=np.int64)
            if row_range is not None:
                d = d[(d >= row_range[0]) & (d < row_range[1])]
            if d.size == 0:
                continue
            keys.append(key)
            lens.append(d.size)
            ids.append(np.sort(d) - id_base)
        order = np.argsort(np.asarray(keys, dtype=np.int64), kind="stable")
        keys_s = np.asarray(keys, dtype=np.int64)[order]
        lens_s = np.asarray(lens, dtype=np.int64)[order]
        docids = np.concatenate([ids[i] for i in order]).astype(np.int32) if len(ids) else np.zeros(0, np.int32)
        offsets = np.zeros(len(keys_s) + 1, dtype=np.int64)
        np.cumsum(lens_s, out=offsets[1:])
        return cls(torch.from_numpy(keys_s).to(dev), torch.from_numpy(offsets).to(dev), torch.from_numpy(docids).to(dev),
                   M, K, id_base)

    def occurrence_table(self):
        """-> (occ int32 [n, C-1], C), built on the device on first use and kept: C is the largest number of leaves that
        list one document (`--doc_multiclus`; 1 for a single-cluster index, whose table is empty), and row p of occ
        holds the CSR leaf indices of the document's other positions, -1 padded (-2 - leaf for an earlier position in
        the same leaf: a leaf that lists the document twice)."""
        if self._occ is None:
            self._occ = _lib.get_context(self.device.index).occurrence_table(self.leaf_offsets, self.leaf_docids)
        return self._occ

    # -- queries --------------------------------------------------------------
    def lookup(self, dec) -> torch.Tensor:
        """Beam-search leaves [nq, L, M] (any int dtype, host or device) -> CSR leaf index int32
        [nq, L], -1 where the leaf holds no document (`doc_cluster.get(d, None)`, 3928)."""
        if not isinstance(dec, torch.Tensor):
            dec = torch.from_numpy(np.asarray(dec))
        dec = dec.to(self.device, torch.int64).contiguous()
        if self.n_leaves == 0 or dec.numel() == 0:
            return torch.full(dec.shape[:-1], -1, dtype=torch.int32, device=self.device)
        return _lib.get_context(self.device.index).leaf_lookup(dec, self.K, self.leaf_keys)

    # -- reference-format dictionaries ---------------------------------------
    def to_dicts(self):
        """(rqclus, rqmapping) python dictionaries in the reference's format and ORDER (global doc ids): leaves in order
        of first appearance (= ascending smallest doc id, pq.py:236-242), doc ids ascending inside a leaf, mapping in doc
        order - `pickle.dumps` of either equals the reference's file byte for byte.  One D2H copy of the CSR, numpy
        grouping, python objects via tolist(); the only interpreter loop runs over the leaves."""
        keys = self.leaf_keys.cpu().numpy()
        offs = self.leaf_offsets.cpu().numpy()
        local = self.leaf_docids.cpu().numpy().astype(np.int64)
        n, nl = local.shape[0], keys.shape[0]
        digits = np.zeros((nl, self.M), dtype=np.int64)
        k = keys.copy()
        for j in range(self.M - 1, -1, -1):
            digits[:, j] = k % self.K
            k //= self.K
        leaf_of_pos = np.repeat(np.arange(nl), np.diff(offs))
        codes = np.empty((n, self.M), dtype=np.int64)
        codes[local] = digits[leaf_of_pos]                      # code tuple of every local row
        tuples = list(map(tuple, codes.tolist()))
        mapping = dict(zip(range(self.id_base, self.id_base + n), tuples))
        first_doc = local[offs[:-1]] if nl else np.zeros(0, np.int64)
        docs = local + self.id_base
        cluster = {}
        for g_ in np.argsort(first_doc, kind="stable").tolist():
            cluster[tuples[first_doc[g_]]] = docs[offs[g_] : offs[g_ + 1]].tolist()
        return cluster, mapping



# ---- leaf-grouped (tensor-core) re-rank: host-side planning ------------------------------------------------
GROUP_COLS = 64      # queries per GEMM column group (GR_TN in csrc/flat_tensor.cu)
TILE_ROWS = 128      # document rows per GEMM tile (UMMA M)


def build_leaf_tiles(leaf_offsets: torch.Tensor):
    """Tiles of TILE_ROWS rows of the leaf-ordered matrix that never straddle a leaf.
    -> (tile_row0 int32 [T], tile_nrows int32 [T], leaf_tile0 int64 [n_leaves+1], src_index int32 [T*128], -1 = padding)."""
    off = leaf_offsets.to(torch.int64)
    dev = off.device
    sizes = off[1:] - off[:-1]
    tpl = (sizes + TILE_ROWS - 1) // TILE_ROWS
    leaf_tile0 = torch.zeros(off.numel(), dtype=torch.int64, device=dev)
    torch.cumsum(tpl, 0, out=leaf_tile0[1:])
    T = int(leaf_tile0[-1].item())
    tile_leaf = torch.repeat_interleave(torch.arange(sizes.numel(), device=dev), tpl)
    local = torch.arange(T, device=dev) - leaf_tile0[tile_leaf]
    row0 = off[tile_leaf] + local * TILE_ROWS
    nrows = torch.minimum(off[tile_leaf + 1] - row0, torch.full_like(row0, TILE_ROWS))
    r = torch.arange(TILE_ROWS, device=dev)
    src = row0[:, None] + r[None, :]
    src = torch.where(r[None, :] < nrows[:, None], src, torch.full_like(src, -1))
    return (row0.to(torch.int32).contiguous(), nrows.to(torch.int32).contiguous(), leaf_tile0,
            src.to(torch.int32).reshape(-1).contiguous())


def plan_grouped_rounds(leaf_offsets: torch.Tensor, leaf_tile0: torch.Tensor, ql: torch.Tensor, round_rows: Sequence[int],
                        bootstrap_rows: int = 0):
    """(leaf, query) pairs of `ql` [nq, L] (CSR leaf index, -1 = none) -> per round the work of the grouped GEMM.

    A pair belongs to round r when the candidate rows listed BEFORE it in its query's leaf list number less than
    round_rows[r] (and not less than round_rows[r-1]); the last round takes the rest.  With `bootstrap_rows` > 0 a
    round is put in front of these: the leading pairs of every query whose candidate rows, the pair's own leaf
    INCLUDED, number at most bootstrap_rows - the round that runs without thresholds (every score is appended), so it
    must fit the candidate buffers by construction.  Per round: pairs sorted by leaf, each leaf's queries cut into
    groups of GROUP_COLS columns, one work item per (tile of the leaf, group).
    -> list of (item_tile int32 [I], item_group int32 [I], group_qid int32 [G*GROUP_COLS], -1 = padding)."""
    dev = ql.device
    off = leaf_offsets.to(torch.int64)
    sizes = off[1:] - off[:-1]
    nq, L = ql.shape
    valid = ql >= 0
    qsz = torch.where(valid, sizes[ql.clamp(min=0).long()], torch.zeros((), dtype=torch.int64, device=dev))
    before = torch.cumsum(qsz, 1) - qsz
    bounds = torch.tensor(list(round_rows), dtype=torch.int64, device=dev)
    rnd = torch.bucketize(before, bounds, right=True)  # rows before < round_rows[0] -> 0, ...
    n_rounds = len(round_rows) + 1
    if bootstrap_rows > 0:
        rnd = torch.where(before + qsz <= bootstrap_rows, torch.zeros_like(rnd), rnd + 1)
        n_rounds += 1
    qidx = torch.arange(nq, device=dev)[:, None].expand(nq, L)
    tpl = leaf_tile0[1:] - leaf_tile0[:-1]
    out = []
    for r in range(n_rounds):
        m = valid & (rnd == r)
        leaf = ql[m].long()
        q = qidx[m]
        if leaf.numel() == 0:
            out.append((torch.zeros(0, dtype=torch.int32, device=dev),) * 2 + (torch.zeros(0, dtype=torch.int32, device=dev),))
            continue
        order = torch.argsort(leaf, stable=True)
        leaf, q = leaf[order], q[order]
        uleaf, cnt = torch.unique_consecutive(leaf, return_counts=True)
        run0 = torch.cumsum(cnt, 0) - cnt                                   # first pair of every leaf run
        gpl = (cnt + GROUP_COLS - 1) // GROUP_COLS                          # groups per leaf
        grp0 = torch.cumsum(gpl, 0) - gpl
        G = int(gpl.sum().item())
        run_of_pair = torch.repeat_interleave(torch.arange(uleaf.numel(), device=dev), cnt)
        pos = torch.arange(leaf.numel(), device=dev) - run0[run_of_pair]
        grp_of_pair = grp0[run_of_pair] + pos // GROUP_COLS
        group_qid = torch.full((G, GROUP_COLS), -1, dtype=torch.int32, device=dev)
        group_qid[grp_of_pair, pos % GROUP_COLS] = q.to(torch.int32)
        # work items, per leaf TILE-major: a document tile (196 KB) comes from HBM once and meets all the query groups of
        # its leaf back to back; the groups' images (98 KB each) are what gets re-read, and they stay in L2
        ntl = tpl[uleaf]
        ipl = ntl * gpl                                                     # items per leaf
        item0 = torch.cumsum(ipl, 0) - ipl
        leaf_of_item = torch.repeat_interleave(torch.arange(uleaf.numel(), device=dev), ipl)
        local = torch.arange(leaf_of_item.numel(), device=dev) - item0[leaf_of_item]
        g_of = gpl[leaf_of_item]
        item_tile = leaf_tile0[uleaf[leaf_of_item]] + local // g_of
        item_group = grp0[leaf_of_item] + local % g_of
        out.append((item_tile.to(torch.int32).contiguous(), item_group.to(torch.int32).contiguous(),
                    group_qid.reshape(-1).contiguous()))
    return out


class ClusterReranker:
    """Holds a (shard of the) doc-embedding matrix on the device plus its inverted lists."""

    AUTO_MIN_DOCS = 1 << 18         # mode='auto': corpora below this stay on the streaming kernel (no tile image)
    AUTO_QUERIES_PER_LEAF = 4       # mode='auto': grouped path when nq*L >= this many (query, leaf) pairs per leaf
    AUTO_ALL_QUERIES_PER_LEAF = 0.25  # rerank_all, mode='auto': grouped scorer from this many (query, leaf) pairs per
                                      # leaf.  Scoring at L = 10, 8.8 M x 768 (B200, 1,000 W): 0.12 pairs per leaf
                                      # 4.3 ms stream / 4.8 ms grouped, 0.24: 7.8 / 7.5, 0.49: 14.7 / 10.2, 3.0: 75 / 23
    BOOTSTRAP_ROWS = 3072           # rows of the threshold-free first round per query (all appended: must fit the buffers)
    BOOTSTRAP_MIN = 2048            # fewer bootstrap rows than this: first threshold from the streaming kernel instead ...
    PASS_BUDGET = 6144              # ... unless the query has so few candidates that its sample's k-th best lets fewer than
                                    # this many (of the 8,192 buffer slots) through the last round: a sample of s rows
                                    # passes ~candidates * k / s
    ROUND_ROWS = (32768,)           # pairs whose preceding candidate rows number less than this go first
    PLAN = "device"                 # "device": the tiles plan made by the library (mevi_rerank_grouped_plan; default);
                                    # "tiles": its torch restatement plan_grouped_tile_rounds; "prefix": plan_grouped_rounds
    SHARE_THRESHOLDS = False        # sharded documents: all-reduce(MAX) of the thresholds after every round.  Correct and
                                    # tested (tests/dist_check.py), but measured slower (5.26 vs 5.13 ms per call at N = 4:
                                    # the sharded call is bound by launches and per-query kernels, not by the candidates
                                    # the shared bound removes): opt-in, MEVI_RERANK_SHARE=1
    MAXG_SAMPLE = 1                 # query groups (of 64) an item of a sample round takes
    MAXG_LAST = 4                   # ... and of the last round: a document tile is fetched once for up to 256 queries
    BOOT_LEAVES = (8, 128)          # tiles plan: first tile of the leading 8 leaves = the threshold-free bootstrap (<= 1,024
                                    # appended rows per query), then the first tile of the next 120 (= of ALL the leaves at
                                    # the shipped L = 100) filtered by it; the last round is left with the further tiles.
                                    # Measured at 6,980 x 100: (8, 100) 6.9 ms, (8, 63) 7.6, (8, 40) 8.2, (8, 32, 100) 7.3

    def __init__(self, all_embeddings, index: ClusterIndex, device_index: Optional[int] = None,
                 leaf_ordered: bool = True, mode: Optional[str] = None, D_leaf: Optional[torch.Tensor] = None):
        """`leaf_ordered=True` (default) keeps a copy of the matrix permuted into CSR order so that each
        leaf is one contiguous byte range (streamed with bulk async copies); False gathers candidate
        rows one by one from the document-ordered matrix."""
        self.ctx = _lib.get_context(device_index if device_index is not None else index.device.index)
        dev = torch.device("cuda", self.ctx.device)
        if D_leaf is not None:  # the caller already holds the leaf-ordered copy (ctx.gather_rows(D, index.leaf_docids))
            D = None
        elif isinstance(all_embeddings, torch.Tensor):
            D = all_embeddings.to(device=dev, dtype=torch.float32).contiguous()
        else:
            from .trainer import _upload_rows

            D = _upload_rows(all_embeddings, 0, all_embeddings.shape[0], dev)
        self.index = index
        self.leaf_ordered = bool(leaf_ordered)
        if D_leaf is not None:
            assert leaf_ordered and D_leaf.is_cuda and D_leaf.dtype == torch.float32 and D_leaf.is_contiguous()
            self.D = D_leaf
        else:
            self.D = self.ctx.gather_rows(D, index.leaf_docids) if self.leaf_ordered else D
        # "stream": one pass over every query's candidates (rerank.cu); "grouped": every leaf read once and scored against
        # all the queries that chose it on the tensor cores (flat_tensor.cu, K3g), falling back to "stream" per call when
        # the prefilter guarantee cannot be established
        import os

        # "auto" (default): build the tile image when the corpus is large enough for leaf sharing to matter and it fits, and
        # take the grouped path per call when the queries share leaves (>= AUTO_QUERIES_PER_LEAF (query, leaf) pairs per leaf)
        self.mode = mode or os.environ.get("MEVI_RERANK_MODE", "auto")
        if self.mode not in ("stream", "grouped", "auto"):
            raise ValueError(f"unknown re-rank mode {self.mode!r}")
        self._grouped = None
        self.last_path = None
        if os.environ.get("MEVI_RERANK_BOOTSTRAP"):
            self.BOOTSTRAP_ROWS = int(os.environ["MEVI_RERANK_BOOTSTRAP"])
        if os.environ.get("MEVI_RERANK_SHARE"):
            self.SHARE_THRESHOLDS = os.environ["MEVI_RERANK_SHARE"] != "0"
        if os.environ.get("MEVI_RERANK_PLAN"):
            self.PLAN = os.environ["MEVI_RERANK_PLAN"]
        if os.environ.get("MEVI_RERANK_MAXG"):
            self.MAXG_LAST = int(os.environ["MEVI_RERANK_MAXG"])
        if os.environ.get("MEVI_RERANK_ROUNDS"):
            self.ROUND_ROWS = tuple(int(v) for v in os.environ["MEVI_RERANK_ROUNDS"].split(","))
        build_image = self.mode == "grouped"
        if self.mode == "grouped" and not self.leaf_ordered:
            raise ValueError("mode='grouped' needs the leaf-ordered layout")
        if self.mode == "auto" and self.leaf_ordered and self.D.shape[0] >= self.AUTO_MIN_DOCS and self.D.shape[1] % 64 == 0:
            n_leaves = int(index.leaf_offsets.numel()) - 1
            img_bytes = (self.D.shape[0] + 128 * n_leaves) * self.D.shape[1] * 2  # upper bound incl. per-leaf padding
            build_image = torch.cuda.mem_get_info(dev)[0] >= 2 * img_bytes + (4 << 30)
        if build_image:
            row0, nrows, leaf_tile0, src = build_leaf_tiles(index.leaf_offsets)
            img, absmax, maxnorm = self.ctx.rerank_grouped_image(self.D, src, row0.numel())
            del src
            self._grouped = dict(row0=row0, nrows=nrows, leaf_tile0=leaf_tile0, img=img, absmax=absmax, maxnorm=maxnorm)

    @torch.no_grad()
    def rerank(self, query_embedding, dec, topk: int = 100, multiclus_score_aggr: Optional[str] = None):
        """-> (scores [nq,k] fp32 desc, ids [nq,k] int64 (-1 padded), n_candidates [nq] int32), on the device.
        With torch.distributed initialised the documents are sharded: every rank scores the
        candidates it owns, the per-shard lists are all-gathered and merged on every rank.

        `multiclus_score_aggr` in ('add', 'max') is the `--doc_multiclus > 1` top-k (main_models.py:3998-4011, then the
        sort and `[:save_hard_neg]`) for an index that lists a document under up to C <= 16 leaves.  For a query and a
        document, c = the number of positions of the query's leaf list whose leaf lists the document (a repeated leaf
        counts once per position, and a leaf listing the document twice counts twice, like the reference's concatenation)
        and s = its fp32 score, the same at every
        position.  The document appears once, scored s ('max') or by the fp32 fold ((0 + s) + s) + ... of c terms
        ('add', the reference's order; for c <= 2 it equals rerank_all's scatter_add_ bit for bit).  The k best
        distinct documents by (score desc, id asc), rerank_all's order; n_candidates counts occurrences (cur_ndoc).
        The streaming kernel keeps only the occurrence at the earliest position of the leaf list and scores it
        agg(c, s) (last_path = "stream-multiclus").  Row-block shards (`from_cluster_dict(row_range=...)`) keep every
        occurrence of a document on one rank, so the all-gather + merge stays exact; a leaf-partitioned shard
        (index.doc_ids set) can hold a document's other leaves on other ranks and raises NotImplementedError.
        None: the single-cluster path, unchanged."""
        dev = self.D.device
        if not isinstance(query_embedding, torch.Tensor):
            query_embedding = torch.from_numpy(np.ascontiguousarray(query_embedding, dtype=np.float32))
        Q = query_embedding.to(device=dev, dtype=torch.float32).contiguous()
        if multiclus_score_aggr is not None:
            return self._rerank_multiclus(Q, dec, topk, multiclus_score_aggr)
        ql = self.index.lookup(dec)
        use_grouped = self._grouped is not None and (
            self.mode == "grouped" or ql.numel() >= self.AUTO_QUERIES_PER_LEAF * max(1, self.index.n_leaves))
        # threshold sharing is a collective inside the grouped path: it runs only when EVERY rank takes that path for this
        # call (the ranks decide independently: shard size, image fits, leaves shared), agreed on by one all-reduce(MIN)
        self._share_now = False
        if dist_on() and self.SHARE_THRESHOLDS:
            mine = use_grouped and self._grouped["absmax"] >= 0 and topk <= 256 and Q.shape[0] > 0 and self.PLAN in ("device", "tiles")
            flag = torch.tensor([1 if mine else 0], dtype=torch.int32, device=dev)
            torch.distributed.all_reduce(flag, op=torch.distributed.ReduceOp.MIN)
            self._share_now = bool(flag.item())
        out = self._rerank_grouped(Q, ql, topk) if use_grouped else None
        if out is None:
            self.last_path = "stream"
            out = self.ctx.cluster_rerank(Q, self.D, self.index.leaf_offsets, self.index.leaf_docids, ql, topk,
                                          id_base=self.index.id_base, leaf_ordered=self.leaf_ordered)
        scores, ids, ncand = out
        if self.index.doc_ids is not None:  # leaf-partitioned shard: local rows -> document ids
            ids = torch.where(ids >= 0, self.index.doc_ids[(ids - self.index.id_base).clamp(min=0)], ids)
        if dist_on():
            s_all = all_gather_stack(scores)
            i_all = all_gather_stack(ids)
            scores, ids = self.ctx.topk_merge(s_all.contiguous(), i_all.contiguous())
            torch.distributed.all_reduce(ncand)
        return scores, ids, ncand


def _rerank_multiclus(self, Q, dec, topk, aggr):
    if aggr not in ("add", "max"):
        raise ValueError("multiclus_score_aggr must be 'add' or 'max' (main_models.py:4002-4009)")
    if self.index.doc_ids is not None:
        raise NotImplementedError("multi-cluster re-rank on a leaf-partitioned shard: a document's other leaves can live "
                                  "on other ranks")
    if not self.leaf_ordered:
        raise ValueError("multi-cluster re-rank needs the leaf-ordered layout")
    idx = self.index
    occ, n_occ = idx.occurrence_table()
    ql = idx.lookup(dec)
    # the grouped path under the single-cluster call's conditions (mode, pairs per leaf; _rerank_grouped: image, topk)
    use_grouped = self._grouped is not None and n_occ <= 16 and ql.shape[1] <= 4096 and (
        self.mode == "grouped" or ql.numel() >= self.AUTO_QUERIES_PER_LEAF * max(1, idx.n_leaves))
    out = self._rerank_grouped(Q, ql, topk, multiclus=(occ, n_occ, aggr)) if use_grouped else None
    if out is None:
        out = self.ctx.cluster_rerank_multiclus(Q, self.D, idx.leaf_offsets, idx.leaf_docids, occ, n_occ, ql, topk, aggr,
                                                id_base=idx.id_base)
        self.last_path = "stream-multiclus"
    scores, ids, ncand = out
    if dist_on():
        scores, ids = self.ctx.topk_merge(all_gather_stack(scores).contiguous(), all_gather_stack(ids).contiguous())
        torch.distributed.all_reduce(ncand)
    return scores, ids, ncand


ClusterReranker._rerank_multiclus = _rerank_multiclus


@torch.no_grad()
def _rerank_all(self, query_embedding, dec, multiclus_score_aggr: Optional[str] = None):
    """The shipped recipe's output mode (`--save_hard_neg <corpus size>`, main_models.py:4012-4014, 4046-4053): EVERY
    candidate of every query, sorted by score descending, as a CSR over the queries:
        -> (offsets int64 [nq+1], ids int64 [total], scores fp32 [total]) on the device.
    `multiclus_score_aggr` in ('add', 'max') is the `--doc_multiclus > 1` aggregation of 3998-4011: a document listed
    under several of the query's leaves appears once, with its scores added or maximised (`np.unique` + loop there).
    Scores come from `mevi_cluster_rerank_all` (mode "stream": one pass over every query's candidates) or
    `mevi_cluster_rerank_all_grouped` (mode "grouped": every leaf read once for all the queries that chose it; "auto"
    takes it with at least AUTO_ALL_QUERIES_PER_LEAF (query, leaf) pairs per leaf of the index); both give the dense
    scorer's summation order bit for bit (equal to the top-k paths), and `last_path` says which ran ("grouped-all" /
    "stream-all").  The sort is `mevi_sort_candidates`, a segmented device sort (sort_candidates_torch restates it),
    ties ordered by ascending doc id (the reference's CUDA `torch.sort` leaves tie order unspecified).  `--knn_topk_by_step` (3986-3989, a running top-pool_size) is `rerank(topk=pool_size)`.
    A leaf-partitioned shard (index.doc_ids set) maps its rows to document ids before the sort, so ties are ordered by
    the document id.
    With torch.distributed initialised the documents are sharded: every rank sorts its own candidates as above, the
    per-rank CSRs are all-gathered and `mevi_merge_sorted_runs` merges the sorted runs, so every rank returns the whole
    corpus's answer - bit-identical to the single-GPU call on the whole index: a candidate's score is computed from the
    same row in the same order on whichever rank owns it, and (score, id) orders the candidates of different ranks
    totally.  With 'add' and a document under c >= 3 of the query's leaves the single-GPU fold order is unspecified
    (scatter_add_), so such scores agree within that rounding.  A multi-cluster call on a leaf-partitioned shard raises
    NotImplementedError (a document's other leaves can live on other ranks); at most 8 ranks.  Extra device memory per
    rank: the gathered runs and the output, 12 bytes per candidate of the whole corpus each, plus one more such buffer
    with more than 2 ranks (the merge passes' intermediate)."""
    if not self.leaf_ordered:
        raise ValueError("rerank_all needs the leaf-ordered layout")
    if multiclus_score_aggr is not None and multiclus_score_aggr not in ("add", "max"):
        raise ValueError("multiclus_score_aggr must be 'add' or 'max' (main_models.py:4002-4009)")
    idx = self.index
    if multiclus_score_aggr is not None and idx.doc_ids is not None:
        raise NotImplementedError("multi-cluster rerank_all on a leaf-partitioned shard: a document's other leaves can "
                                  "live on other ranks")
    world = rank_world()[1]
    if world > 8:
        raise NotImplementedError(f"rerank_all under torch.distributed merges at most 8 ranks (world size {world})")
    dev = self.D.device
    if not isinstance(query_embedding, torch.Tensor):
        query_embedding = torch.from_numpy(np.ascontiguousarray(query_embedding, dtype=np.float32))
    Q = query_embedding.to(device=dev, dtype=torch.float32).contiguous()
    ql = idx.lookup(dec)
    on_device = self.D.is_cuda
    grouped = False
    if on_device:  # the scorer: every leaf read once for all its queries, or one pass per query (the same bits)
        grouped = self.mode == "grouped" or (
            self.mode == "auto" and ql.numel() >= self.AUTO_ALL_QUERIES_PER_LEAF * max(1, idx.n_leaves))
        self.last_path = "grouped-all" if grouped else "stream-all"
        offsets, scores, ids, _ = self.ctx.cluster_rerank_all(Q, self.D, idx.leaf_offsets, idx.leaf_docids, ql,
                                                              id_base=idx.id_base, grouped=grouped)
    else:
        offsets, scores, ids, _ = self.ctx.cluster_rerank_all(Q, self.D, idx.leaf_offsets, idx.leaf_docids, ql,
                                                              id_base=idx.id_base)
    if idx.doc_ids is not None:  # leaf-partitioned shard: local rows -> document ids (id_base is 0 there)
        ids = idx.doc_ids[ids]
    nq = Q.shape[0]
    seg = None
    if multiclus_score_aggr is not None:
        seg = torch.repeat_interleave(torch.arange(nq, device=dev), offsets[1:] - offsets[:-1])
        span = int(ids.max().item()) + 1 if ids.numel() else 1
        key, inv = torch.unique(seg * span + ids, return_inverse=True)
        agg = torch.zeros(key.numel(), dtype=torch.float32, device=dev)
        if multiclus_score_aggr == "add":
            agg.scatter_add_(0, inv, scores)
        else:
            agg.fill_(float("-inf")).scatter_reduce_(0, inv, scores, reduce="amax")
        seg, ids, scores = key // span, key % span, agg
        counts = torch.bincount(seg, minlength=nq)
        offsets = torch.zeros(nq + 1, dtype=torch.int64, device=dev)
        torch.cumsum(counts, 0, out=offsets[1:])
    if on_device:  # mevi_sort_candidates, in place
        scores, ids = self.ctx.sort_candidates(offsets, scores, ids, out=(scores, ids))
    else:
        scores, ids = sort_candidates_torch(offsets, scores, ids)
    del seg
    if not dist_on():
        return offsets, ids, scores
    # every rank's sorted CSR to every rank (one block per rank), then one merge of the sorted runs
    run_offsets = all_gather_stack(offsets)
    gathered_scores = all_gather_varlen(scores)
    del scores
    gathered_ids = all_gather_varlen(ids)
    del ids
    run_len = run_offsets[:, -1]
    bases = torch.cumsum(run_len, 0) - run_len
    out_offsets = run_offsets.sum(0)
    scores, ids = self.ctx.merge_sorted_runs(gathered_scores, gathered_ids, bases, run_offsets, out_offsets)
    return out_offsets, ids, scores


def sort_candidates_torch(offsets, scores, ids):
    """Every query's segment of a CSR sorted by (score desc, id asc) through three stable torch passes, least significant
    key first: the restatement of `mevi_sort_candidates` (Context.sort_candidates), and rerank_all's sort on CPU tensors.
    -> (scores, ids)."""
    nq = offsets.numel() - 1
    seg = torch.repeat_interleave(torch.arange(nq, device=offsets.device), offsets[1:] - offsets[:-1])
    order = torch.argsort(ids, stable=True)
    order = order[torch.argsort(scores[order], descending=True, stable=True)]
    order = order[torch.argsort(seg[order], stable=True)]
    return scores[order], ids[order]


def hn_lines_all(texts: Sequence[str], offsets, ids, scores, save_hard_neg: Optional[int] = None,
                 gt_outputs: Optional[Sequence[str]] = None) -> List[str]:
    """hn lines (main_models.py:4046-4053) from the CSR of `rerank_all`: all candidates, truncated to
    `[:save_hard_neg]` like the reference's slices."""
    off = offsets.cpu().numpy()
    i = ids.cpu().numpy()
    s = scores.cpu().numpy()
    lines = []
    for r, text in enumerate(texts):
        a, b = int(off[r]), int(off[r + 1])
        if save_hard_neg is not None:
            b = min(b, a + int(save_hard_neg))
        docs = ",".join(str(int(x)) for x in i[a:b])
        sc = ",".join(str(float(x)) for x in s[a:b])
        gt = gt_outputs[r] if gt_outputs is not None else ""
        lines.append("\t".join([text, gt, docs, sc]))
    return lines


ClusterReranker.rerank_all = _rerank_all


def _group_items(leaf, q, first_tile, n_tiles, presorted: bool = False, maxg: int = 1):
    """Work items of one item set: (leaf, query) pairs (1-D; sorted by leaf when `presorted`) meet the tiles
    [first_tile[leaf], first_tile[leaf] + n_tiles[leaf]) of their leaf.  Each leaf's queries are cut into groups of
    GROUP_COLS columns, one item per (tile, group), per leaf TILE-major: a document tile (196 KB) comes from HBM once and
    meets all the query groups of its leaf back to back.
    An item takes up to `maxg` consecutive groups of its leaf (item_group = first group | number of groups << 24).
    -> (item_tile int32 [I], item_group int32 [I], group_qid int32 [G*GROUP_COLS]).  One host sync (G and I)."""
    dev = leaf.device
    keep = n_tiles[leaf] > 0
    leaf, q = leaf[keep], q[keep]
    if leaf.numel() == 0:
        z = torch.zeros(0, dtype=torch.int32, device=dev)
        return z, z, z
    if not presorted:
        order = torch.argsort(leaf, stable=True)
        leaf, q = leaf[order], q[order]
    uleaf, cnt = torch.unique_consecutive(leaf, return_counts=True)
    run0 = torch.cumsum(cnt, 0) - cnt                                   # first pair of every leaf run
    gpl = (cnt + GROUP_COLS - 1) // GROUP_COLS                          # groups per leaf
    grp0 = torch.cumsum(gpl, 0) - gpl
    wpl = (gpl + maxg - 1) // maxg                                      # wide items per tile of the leaf
    ipl = n_tiles[uleaf] * wpl                                          # items per leaf
    G, n_items = (int(v) for v in torch.stack([gpl.sum(), ipl.sum()]).tolist())
    run_of_pair = torch.repeat_interleave(torch.arange(uleaf.numel(), device=dev), cnt, output_size=leaf.numel())
    pos = torch.arange(leaf.numel(), device=dev) - run0[run_of_pair]
    grp_of_pair = grp0[run_of_pair] + pos // GROUP_COLS
    group_qid = torch.full((G, GROUP_COLS), -1, dtype=torch.int32, device=dev)
    group_qid[grp_of_pair, pos % GROUP_COLS] = q.to(torch.int32)
    item0 = torch.cumsum(ipl, 0) - ipl
    leaf_of_item = torch.repeat_interleave(torch.arange(uleaf.numel(), device=dev), ipl, output_size=n_items)
    local = torch.arange(n_items, device=dev) - item0[leaf_of_item]
    w_of = wpl[leaf_of_item]
    item_tile = first_tile[uleaf[leaf_of_item]] + local // w_of
    j = (local % w_of) * maxg
    item_group = grp0[leaf_of_item] + j
    if maxg > 1:
        item_group = item_group | (torch.clamp(gpl[leaf_of_item] - j, max=maxg) << 24)
    return item_tile.to(torch.int32).contiguous(), item_group.to(torch.int32).contiguous(), group_qid.reshape(-1).contiguous()


def plan_grouped_tile_rounds(leaf_tile0: torch.Tensor, ql: torch.Tensor, boot_leaves, maxg_sample: int = 1, maxg_last: int = 1):
    """Rounds that cut the work by TILES instead of by leaf prefixes, so that a leaf's queries stay together.  With
    boot_leaves = (b0, b1, ...):
      round 0 (threshold-free bootstrap): the FIRST tile of the first b0 leaves of every query - at most b0 * TILE_ROWS
              appended scores per query, a sample spread over the query's leaves;
      round i: the first tile of the leaves with rank in [b(i-1), b(i)), filtered by the thresholds of the rounds before
              (appending is the expensive part of a round that passes everything, so the sample grows in two steps);
      last round: the first tile for the pairs the bootstrap left out, and every further tile of every leaf against ALL
              the queries that chose the leaf (full groups: a tile meets ceil(queries / GROUP_COLS) groups once).
    The prefix plan (`plan_grouped_rounds`) splits a leaf's queries over its rounds, so every tile is fetched, and its
    query groups rebuilt, once per round.  -> [(item_tile, item_group, group_qid)] per round.
    This is the torch restatement of csrc/rerank_plan.cu (mevi_rerank_grouped_plan), which the re-ranker uses by default;
    the two agree up to the order of the queries inside a leaf's groups."""
    if isinstance(boot_leaves, int):
        boot_leaves = (boot_leaves,)
    dev = ql.device
    nq, L = ql.shape
    valid = ql >= 0
    tpl = leaf_tile0[1:] - leaf_tile0[:-1]
    first = leaf_tile0[:-1]
    one = torch.clamp(tpl, max=1)
    # all valid pairs sorted by leaf ONCE (stable: queries ascend inside a leaf); the rounds are order-preserving subsets
    leaf_all = ql[valid].long()
    order = torch.argsort(leaf_all, stable=True)
    leaf_all = leaf_all[order]
    q_all = torch.arange(nq, device=dev)[:, None].expand(nq, L)[valid][order]
    rank_all = torch.arange(L, device=dev)[None, :].expand(nq, L)[valid][order]
    out = []
    lo = 0
    for hi in boot_leaves:
        m = (rank_all >= lo) & (rank_all < hi)
        out.append(_group_items(leaf_all[m], q_all[m], first, one, presorted=True, maxg=maxg_sample))
        lo = hi
    m1 = rank_all >= lo
    a_t, a_g, a_q = _group_items(leaf_all[m1], q_all[m1], first, one, presorted=True, maxg=maxg_last)
    b_t, b_g, b_q = _group_items(leaf_all, q_all, first + 1, tpl - one, presorted=True, maxg=maxg_last)
    out.append((torch.cat([a_t, b_t]), torch.cat([a_g, b_g + a_q.numel() // GROUP_COLS]), torch.cat([a_q, b_q])))
    return out


def _rerank_grouped(self, Q, ql, topk, multiclus=None):
    """Leaf-grouped tensor-core path; None when it does not apply or could not establish its guarantee for the call.
    Queries whose own guarantee fails (candidate buffer or margin-window overflow: near-duplicate documents, one huge
    leaf) are re-run through the streaming kernel and patched in; the answer is always the exact one.
    multiclus = (occ, C, aggr): the multi-cluster top-k of _rerank_multiclus (one entry per document, aggregated
    scores; DESIGN §4), bit-equal to mevi_cluster_rerank_multiclus, which re-runs the failed and the weak queries."""
    g = self._grouped
    if g["absmax"] < 0 or topk > 256 or Q.shape[0] == 0:
        return None
    ctx, idx = self.ctx, self.index
    off = idx.leaf_offsets
    boot = (self.BOOT_LEAVES,) if isinstance(self.BOOT_LEAVES, int) else tuple(self.BOOT_LEAVES)
    ql_all = ql
    if multiclus is not None:
        # the multi-cluster state hangs off the call's state (margins, norms): _begin first.  The plan sees one pair per
        # distinct leaf; c and n_candidates count every position of the unmasked list.
        if "tile_leaf" not in g:
            lt0 = g["leaf_tile0"]
            g["tile_leaf"] = torch.repeat_interleave(torch.arange(lt0.numel() - 1, device=lt0.device, dtype=torch.int32),
                                                     lt0[1:] - lt0[:-1]).contiguous()
        ctx.rerank_grouped_begin(Q, g["absmax"], g["maxnorm"], None)
        ql, ncand_mc = ctx.rerank_grouped_multiclus(Q, ql_all.contiguous(), off, multiclus[0], multiclus[1], g["tile_leaf"],
                                                    multiclus[2])
    # thresholds bootstrap themselves: the first round (first tiles of the leading leaves of every query) runs without
    # thresholds and appends every score; its compaction yields each query's first k-th best score, the sample rounds
    # that follow tighten it.  A query whose sample is too small for its candidate count (its k-th best would let more
    # than PASS_BUDGET scores through the last round: few, huge leaves) gets the exact k-th score of its first
    # BOOTSTRAP_MIN candidate ROWS from the streaming kernel instead (cuts through the leaf).
    device_plan = None
    if self.PLAN == "device":  # counts, scans, candidate totals and the weak-sample flags in five launches, one host sync
        ql = ql.contiguous()  # the library keeps the pointer until the last plan_fill of this call
        ncand, weak_flags, device_plan, n_weak = ctx.rerank_grouped_plan(ql, off, g["leaf_tile0"], boot, self.BOOTSTRAP_MIN,
                                                                         topk, self.MAXG_SAMPLE, self.MAXG_LAST, self.PASS_BUDGET)
        weak = torch.nonzero(weak_flags).squeeze(1) if n_weak else weak_flags[:0].long()
    else:
        sizes = off[1:] - off[:-1]
        qsz = torch.where(ql >= 0, sizes[ql.clamp(min=0).long()], torch.zeros((), dtype=torch.int64, device=ql.device))
        ncand = qsz.sum(1)
        if self.PLAN == "tiles":  # bootstrap = first tile of the leading BOOT_LEAVES leaves
            boot_rows = qsz[:, :boot[-1]].clamp(max=TILE_ROWS).sum(1)
        else:
            after = torch.cumsum(qsz, 1)
            boot_rows = torch.where(after <= self.BOOTSTRAP_ROWS, qsz, torch.zeros_like(qsz)).sum(1)
        # a sample of s rows lets ~ncand * k / s candidates through the last round: they must fit the candidate buffers
        need = torch.clamp(ncand * topk // self.PASS_BUDGET, min=2 * topk).clamp(max=self.BOOTSTRAP_MIN)
        weak = torch.nonzero((ncand > self.PASS_BUDGET) & (boot_rows < need) & (ncand > boot_rows)).squeeze(1)
        ncand = ncand.clamp(max=0x7FFFFFFF).to(torch.int32)
    self.last_weak_queries = int(weak.numel())
    if multiclus is not None:
        # the prefix's k-th best OCCURRENCE score is no lower bound of the aggregated k-th best: a weak query gets
        # tau = +inf (the rounds append nothing for it) and is re-run whole through the streaming kernel
        ncand = ncand_mc
        if weak.numel():
            tau = torch.full((Q.shape[0],), float("-inf"), dtype=torch.float32, device=Q.device)
            tau[weak] = float("inf")
            ctx.rerank_grouped_thresholds(Q, tau)
    else:
        tau0 = None
        if weak.numel():
            s0, _, _ = ctx.cluster_rerank_prefix(Q[weak].contiguous(), self.D, off, idx.leaf_docids, ql[weak].contiguous(), topk,
                                                 self.BOOTSTRAP_MIN)
            tau0 = torch.full((Q.shape[0],), float("-inf"), dtype=torch.float32, device=Q.device)
            tau0[weak] = s0[:, topk - 1]
        ctx.rerank_grouped_begin(Q, g["absmax"], g["maxnorm"], tau0)
    def share_thresholds():
        # documents sharded over ranks: the largest of the ranks' k-th best scores bounds the global k-th best from below,
        # so after an all-reduce(MAX) of [nq] floats every rank filters the next round - and re-scores - against it
        if multiclus is None and getattr(self, "_share_now", False):
            tau = ctx.rerank_grouped_thresholds(Q)
            torch.distributed.all_reduce(tau, op=torch.distributed.ReduceOp.MAX)
            ctx.rerank_grouped_thresholds(Q, tau)

    if device_plan is not None:
        for r, (n_items, n_groups) in enumerate(device_plan):
            if n_items and n_groups:
                maxg = self.MAXG_LAST if r == len(device_plan) - 1 else self.MAXG_SAMPLE
                item_tile, item_group, group_qid = ctx.rerank_grouped_plan_fill(r, n_items, n_groups, Q.device)
                ctx.rerank_grouped_round(Q, g["img"], g["row0"], g["nrows"], item_tile, item_group, group_qid, topk, maxg)
            share_thresholds()  # every rank, every round (a rank without work in a round still takes part)
    else:
        plan = (plan_grouped_tile_rounds(g["leaf_tile0"], ql, boot, self.MAXG_SAMPLE, self.MAXG_LAST) if self.PLAN == "tiles"
                else plan_grouped_rounds(off, g["leaf_tile0"], ql, self.ROUND_ROWS, self.BOOTSTRAP_ROWS))
        for r, (item_tile, item_group, group_qid) in enumerate(plan):
            if item_tile.numel():
                maxg = 1 if self.PLAN != "tiles" else (self.MAXG_LAST if r == len(plan) - 1 else self.MAXG_SAMPLE)
                ctx.rerank_grouped_round(Q, g["img"], g["row0"], g["nrows"], item_tile, item_group, group_qid, topk, maxg)
            if self.PLAN == "tiles":  # (the prefix plan's number of rounds can differ between ranks)
                share_thresholds()
    nq = Q.shape[0]
    if multiclus is not None:
        scores, ids, failed, n_failed = ctx.rerank_grouped_finish_multiclus(Q, self.D, topk, idx.leaf_docids, idx.id_base)
        self.last_failed_queries = n_failed
        if n_failed >= nq or n_failed > max(16, nq // 4):
            return None
        self.last_path = "grouped-multiclus"
        if n_failed > 0 or weak.numel():
            rerun = failed != 0
            rerun[weak] = True
            bad = torch.nonzero(rerun).squeeze(1)
            s2, i2, _ = ctx.cluster_rerank_multiclus(Q[bad].contiguous(), self.D, off, idx.leaf_docids, multiclus[0], multiclus[1],
                                                     ql_all[bad].contiguous(), topk, multiclus[2], id_base=idx.id_base)
            scores[bad] = s2
            ids[bad] = i2
            self.last_path = "grouped-multiclus+stream"
        return scores, ids, ncand
    scores, rows, failed, n_failed = ctx.rerank_grouped_finish(Q, self.D, topk)
    self.last_failed_queries = n_failed
    if n_failed >= nq or n_failed > max(16, nq // 4):
        return None
    self.last_path = "grouped"
    ids = torch.where(rows >= 0, idx.leaf_docids[rows.clamp(min=0)].to(torch.int64) + idx.id_base, torch.full_like(rows, -1))
    if n_failed > 0:
        bad = torch.nonzero(failed).squeeze(1)
        s2, i2, _ = ctx.cluster_rerank(Q[bad].contiguous(), self.D, off, idx.leaf_docids, ql[bad].contiguous(), topk,
                                       id_base=idx.id_base, leaf_ordered=True)
        scores[bad] = s2
        ids[bad] = i2
        self.last_path = "grouped+stream"
    return scores, ids, ncand


ClusterReranker._rerank_grouped = _rerank_grouped


def hn_lines(texts: Sequence[str], scores, ids, gt_outputs: Optional[Sequence[str]] = None) -> List[str]:
    """The hard-negative / fine result lines of main_models.py:4046-4053 (LogTxtFile joins the
    four fields with tabs, 254-257): query, gt scores, 'd1,d2,...', 's1,s2,...' where each score
    is str(tensor.item()) — the fp32 value widened to a python float."""
    s = scores.detach().cpu().numpy() if isinstance(scores, torch.Tensor) else np.asarray(scores)
    i = ids.detach().cpu().numpy() if isinstance(ids, torch.Tensor) else np.asarray(ids)
    lines = []
    for r, text in enumerate(texts):
        keep = i[r] >= 0
        docs = ",".join(str(int(x)) for x in i[r][keep])
        sc = ",".join(str(float(x)) for x in s[r][keep])
        gt = gt_outputs[r] if gt_outputs is not None else ""
        lines.append("\t".join([text, gt, docs, sc]))
    return lines


def write_hn_file(path: str, texts, scores, ids, gt_outputs=None) -> None:
    with open(path, "w") as fw:
        for line in hn_lines(texts, scores, ids, gt_outputs):
            print(line, file=fw)


def save_index_files(cluster_path: str, doc_cluster: dict, mapping: dict) -> None:
    """rqclus*.pkl / rqmapping*.pkl exactly as main_models.py:3198-3203 writes them
    (mapping path = cluster path with 'clus' -> 'mapping', 3192-3193)."""
    with open(cluster_path, "wb") as fw:
        pickle.dump(doc_cluster, fw)
    with open(cluster_path.replace("clus", "mapping"), "wb") as fw:
        pickle.dump(mapping, fw)


@torch.no_grad()
def eval_all_documents(query_embedding, all_embeddings, pool_size: int, batch_size: int = 1 << 20,
                       device_index: Optional[int] = None):
    """The `--eval_all_documents` branch of MEVI/main_models.py:3818-3876 (twin tower): the reference walks the
    corpus in blocks of `encode_batch_size`, scores q @ p^T and keeps a running torch.topk pool over the
    concatenation.  Here every block goes through `mevi_flat_ip_topk` (tcgen05 prefilter + exact fp32
    re-score) with `id_base` = the block's first row, and the per-block lists are merged by
    `mevi_topk_merge`.  `all_embeddings` may be a CUDA tensor (scored where it lies), a host tensor or an
    np.ndarray / np.memmap (streamed block by block).  With torch.distributed initialised the rows are
    sharded as pq.py:218-225 and the per-shard pools are all-gathered and merged on every rank.
    Returns (stack_scores [nq, min(pool_size, N)] fp32 descending, sorted_docs int32) on the device,
    like the reference's tensors."""
    ctx = _lib.get_context(device_index)
    dev = torch.device("cuda", ctx.device)
    if not isinstance(query_embedding, torch.Tensor):
        query_embedding = torch.from_numpy(np.ascontiguousarray(query_embedding, dtype=np.float32))
    Q = query_embedding.to(device=dev, dtype=torch.float32).contiguous()
    N = all_embeddings.shape[0]
    rank, world = rank_world()
    start, end = shard_bounds(N, rank, world) if dist_on() else (0, N)
    k = int(min(pool_size, N))
    fan_in = max(2, 16384 // max(k, 1))  # mevi_topk_merge sorts at most 16,384 entries per query
    parts_s, parts_i = [], []
    for a in range(start, end, batch_size):
        b = min(a + batch_size, end)
        if isinstance(all_embeddings, torch.Tensor):
            blk = all_embeddings[a:b].to(device=dev, dtype=torch.float32).contiguous()
        else:
            blk = torch.from_numpy(np.ascontiguousarray(all_embeddings[a:b], dtype=np.float32)).to(dev)
        s, i = ctx.flat_ip_topk(Q, blk, k, id_base=a)
        parts_s.append(s)
        parts_i.append(i)
        if len(parts_s) == fan_in:
            s, i = ctx.topk_merge(torch.stack(parts_s).contiguous(), torch.stack(parts_i).contiguous())
            parts_s, parts_i = [s], [i]
    if not parts_s:
        parts_s = [torch.full((Q.shape[0], k), float("-inf"), device=dev)]
        parts_i = [torch.full((Q.shape[0], k), -1, dtype=torch.int64, device=dev)]
    scores, ids = (parts_s[0], parts_i[0]) if len(parts_s) == 1 else ctx.topk_merge(
        torch.stack(parts_s).contiguous(), torch.stack(parts_i).contiguous())
    if dist_on():
        scores, ids = ctx.topk_merge(all_gather_stack(scores).contiguous(), all_gather_stack(ids).contiguous())
    return scores, ids.to(torch.int32)
