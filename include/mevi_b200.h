/*
 * mevi_b200.h — C ABI of libmevi_b200.so, the B200 (sm_100a) implementation of
 * MEVI's index hot path.
 *
 * The reference (HugoZHL/MEVI) has no FFI of its own: the hot path is Python
 * that calls torch / sklearn / faiss.  Each entry point below replaces one of
 * those call sites; the citation after "replaces:" is the reference file:line
 * whose arithmetic the entry point reproduces.  The Python mirror of the
 * reference interface (mevi_b200/pq.py, faiss_search.py, document_encoder.py,
 * rerank.py) binds these symbols with ctypes; INTEGRATION.md shows the stub a
 * reference maintainer would add.
 *
 * Conventions
 *   - Plain C types only.  All array arguments are DEVICE pointers unless the
 *     name ends in `_host`.  Memory is caller-owned; the library keeps no
 *     pointer past the call.  Scratch memory lives in the context and grows on
 *     demand (never shrinks until mevi_ctx_destroy).
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default
 *     stream).  Calls are asynchronous on that stream unless stated otherwise.
 *   - Return value: 0 on success, negative MEVI_ERR_* otherwise;
 *     mevi_last_error(ctx) then returns a message owned by the context.
 *   - A context is bound to one device and is not re-entrant; different
 *     contexts may be used from different threads.
 *   - Row-major (C order) everywhere; `d` is the embedding width.
 */
#ifndef MEVI_B200_H
#define MEVI_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MEVI_ABI_VERSION 1

#define MEVI_OK 0
#define MEVI_ERR_INVALID (-1)     /* bad argument / unsupported shape */
#define MEVI_ERR_CUDA (-2)        /* a CUDA runtime call failed */
#define MEVI_ERR_UNSUPPORTED (-3) /* requested mode not available for this shape */
#define MEVI_ERR_NOMEM (-4)

#define MEVI_METRIC_L2 0 /* pq.py:130  -sum((a-b)^2), argmax */
#define MEVI_METRIC_IP 1 /* pq.py:126   sum(a*b),     argmax */

#define MEVI_MODE_AUTO 0   /* tensor-core path when the shape allows it, else exact */
#define MEVI_MODE_EXACT 1  /* fp32 direct-form on CUDA cores (also the arbiter of flagged rows) */
#define MEVI_MODE_TENSOR 2 /* tcgen05 split-fp16 prefilter + exact fix-up; error if unsupported */

typedef struct mevi_ctx mevi_ctx;

/* ---- context ----------------------------------------------------------- */
int mevi_abi_version(void);
int mevi_ctx_create(int device, mevi_ctx** out);
void mevi_ctx_destroy(mevi_ctx* ctx);
const char* mevi_last_error(mevi_ctx* ctx);
/* info[0]=SM count, [1]=cc major, [2]=cc minor, [3]=total global memory bytes,
 * [4]=1 if the tcgen05 path is usable on this device (cc 10.x), [5]=L2 bytes,
 * [6]=kernels this context has launched so far (its own kernels; library sorts excluded) */
int mevi_device_info(mevi_ctx* ctx, int64_t info[8]);
/* Synchronise `stream` and report what the asynchronous launches before it found: the pipelined kernels bound every
 * mbarrier wait; a time-out (a protocol bug or a hung copy engine, never seen in normal operation) makes the kernel
 * bail out, overwrite its codes with -1 and set a device error word.  Returns MEVI_ERR_CUDA with a message in that
 * case, MEVI_OK otherwise.  The same condition is also reported by the next call on the context and by every call that
 * synchronises on its own (mevi_rq_encode_host, mevi_flat_ip_topk, mevi_rerank_grouped_finish).                  */
int mevi_ctx_check(mevi_ctx* ctx, void* stream);

/* ---- RQ encode ---------------------------------------------------------- *
 * replaces: MEVI/pq.py:281-305 get_rq_document_cluster (+124-131 compute_scores,
 * 121-122 rq_minus_centroids); also the second copy at
 * dataprocess/msmarco_passage/gen_sampled_to_full.py:65-86.
 * Greedy residual quantisation of n rows against codebook[M][K][d]: per level
 * nearest centroid (lowest index on exact fp32 ties), code written as int32,
 * residual -= centroid after every level.
 *   codes             [n, M] int32 out
 *   residual_or_null  [n, d] fp32 out: the residual after the last level
 *                     (pq.py:304-305 subtracts after every level), or NULL
 *   stats_or_null     int64[8] DEVICE out: [0]=rows re-decided by the exact
 *                     fix-up because their prefilter top-2 gap was inside the
 *                     error bound (tensor mode), [1]=rows processed; rest 0 */
int mevi_rq_encode(mevi_ctx* ctx, const float* X, int64_t n, int d, const float* codebook, int M, int K,
                   int metric, int mode, int32_t* codes, float* residual_or_null, int64_t* stats_or_null,
                   void* stream);

/* Same operation on HOST buffers (the call a drop-in pq.get_document_cluster
 * makes on an np.memmap, pq.py:283): rows are streamed to the device in
 * `chunk_rows` pieces through pinned staging buffers, overlapped with the
 * encode of the previous piece; codes are copied back.  Synchronous.
 * stats_host_or_null: int64[8] host out, same meaning as above.              */
int mevi_rq_encode_host(mevi_ctx* ctx, const float* X_host, int64_t n, int d, const float* codebook_host, int M,
                        int K, int metric, int mode, int32_t* codes_host, int64_t chunk_rows,
                        int64_t* stats_host_or_null);

/* ---- k-means (full-batch Lloyd, shardable) ------------------------------ *
 * replaces: MEVI/pq.py:551-598 (rq branch 582-594; sklearn MiniBatchKMeans on
 * rank 0) with the data-parallel form BASELINE.json asks for; the sums/counts
 * exchange mirrors pq.py:384-397.
 * One pass over the shard R[n,d] (the residual of the level being trained):
 *   assign_out_or_null [n] int32, stride `assign_stride` elements between rows
 *                      (so it can write column j of a [n,M] code table)
 *   sums_counts        [K*d + K] fp32 out (overwritten): per-centroid sums of
 *                      the fp32 rows, then per-centroid counts — ONE buffer so
 *                      a single all-reduce(SUM) combines shards
 *   inertia_or_null    double DEVICE out: sum of squared distances to the
 *                      assigned centroid over this shard                      */
int mevi_kmeans_step(mevi_ctx* ctx, const float* R, int64_t n, int d, const float* centroids, int K, int mode,
                     int32_t* assign_out_or_null, int64_t assign_stride, float* sums_counts,
                     double* inertia_or_null, void* stream);
/* ONE pass over the shard for a whole Lloyd iteration (the north star's "centroid GEMM fused with ... per-centroid
 * sum/count accumulation"): while the tensor kernel assigns the rows to `centroids`, the same streamed tiles are summed
 * per centroid under the rows' PREVIOUS assignment (known before the pass; the new one is only known after a row's
 * last column):
 *   prev_assign [n] int32 (stride prev_stride)   in:  assignment of the previous iteration (values clamped to [0,K))
 *   assign_out  [n] int32 (stride assign_stride) out: nearest centroid now (a different buffer than prev_assign)
 *   sums_counts_prev [K*d + K] fp32              out: per-centroid sums | counts of the rows UNDER prev_assign
 * The caller turns these into the sums under assign_out by adding x to the new and subtracting it from the old
 * centroid for the rows whose assignment changed (few after the first iterations): mevi_b200/trainer.py does that with
 * mevi_gather_rows + mevi_accumulate_by_code, in a fixed order - results are bit-reproducible run to run.
 * MEVI_ERR_UNSUPPORTED for shapes outside K <= 32 (K % 4 == 0), d % 64 == 0, K*d*4 <= ~100 KB, n >= 4096: use
 * mevi_kmeans_step.  replaces: the same lines as mevi_kmeans_step.                                                  */
int mevi_kmeans_step_fused(mevi_ctx* ctx, const float* R, int64_t n, int d, const float* centroids, int K,
                           const int32_t* prev_assign, int64_t prev_stride, int32_t* assign_out, int64_t assign_stride,
                           float* sums_counts_prev, double* inertia_or_null, void* stream);
/* ONE pass over the shard per Lloyd iteration, incremental form: the rows are assigned to `centroids` (the only read of
 * the shard), then the running sums | counts are corrected by the rows whose assignment changed since the previous
 * iteration: sums[new] += x, sums[old] -= x (a few per cent of the rows after the first iterations; cost proportional
 * to their number, no host synchronisation).
 *   prev_assign [n] int32 (stride prev_stride)   in:  assignment the master currently describes
 *   assign_out  [n] int32 (stride assign_stride) out: nearest centroid now (a different buffer than prev_assign)
 *   master_sums_counts [K*d + K] float64 DEVICE  in/out: per-centroid sums | counts under prev_assign on entry, under
 *                      assign_out on return (float64 so that repeated corrections do not drift; initialise it from the
 *                      fp32 buffer of one mevi_kmeans_step / mevi_accumulate_by_code)
 *   sums_counts        [K*d + K] fp32 out: the master rounded to fp32 - the buffer the all-reduce and mevi_kmeans_update take
 *   n_changed_or_null  int32 DEVICE out: number of rows that moved
 * Deterministic (ascending row list, fixed slices, no float atomics).  MEVI_ERR_UNSUPPORTED when K > 256 or K*d*4 > 200 KB.
 * replaces: the same lines as mevi_kmeans_step.                                                                     */
int mevi_kmeans_step_delta(mevi_ctx* ctx, const float* R, int64_t n, int d, const float* centroids, int K, int mode,
                           const int32_t* prev_assign, int64_t prev_stride, int32_t* assign_out, int64_t assign_stride,
                           double* master_sums_counts, float* sums_counts, int32_t* n_changed_or_null,
                           double* inertia_or_null, void* stream);
/* centroids[k] = sums[k]/counts[k] where counts[k] > 0 (others unchanged);
 * n_empty_or_null: int32 DEVICE out = number of empty clusters.              */
int mevi_kmeans_update(mevi_ctx* ctx, const float* sums_counts, int K, int d, float* centroids,
                       int32_t* n_empty_or_null, void* stream);
/* R[i,:] -= centroids[assign[i*assign_stride], :]   replaces: pq.py:591-593  */
int mevi_residual_update(mevi_ctx* ctx, float* R, int64_t n, int d, const float* centroids, int K,
                         const int32_t* assign, int64_t assign_stride, void* stream);

/* sums_counts [K*d + K] fp32 out (overwritten): per-centroid sums of the rows of X under a GIVEN assignment,
 * then the per-centroid counts — the same fused buffer mevi_kmeans_step produces, so one all-reduce combines
 * shards.  replaces: MEVI/pq.py:380-393 (ema_update's one-hot scatter + bmm(one_hot^T, vectors) and
 * one_hot.sum(0)) for one level; assign[i*assign_stride] is row i's code at that level.                    */
int mevi_accumulate_by_code(mevi_ctx* ctx, const float* X, int64_t n, int d, const int32_t* assign,
                            int64_t assign_stride, int K, float* sums_counts, void* stream);

/* ---- product-quantiser encode ------------------------------------------- *
 * replaces: MEVI/pq.py:249-279 get_pq_document_cluster ('pq'; 'opq' after the caller applied the rotation of
 * pq.py:259-261).  codebook [M, K, d/M]; codes [n, M] int32 out: per sub-vector j the argmax over k of
 * compute_scores(X[:, j*dsub:(j+1)*dsub], codebook[j,k]) (pq.py:124-131), lowest index on exact fp32 ties. */
int mevi_pq_encode(mevi_ctx* ctx, const float* X, int64_t n, int d, const float* codebook, int M, int K, int metric,
                   int32_t* codes, void* stream);

/* ---- RQ beam search (leaf producer) -------------------------------------- *
 * replaces: MEVI/pq.py:613-713 beam_search, rq branch, do_sample=False: per level
 * softmax_k(compute_scores(residual_b, codebook[i,k])), multiplied by the running beam score when `prod`
 * (rq_topk_score == 'prod'), top-num_beams over beam x K (all candidates kept, in (beam, k) order, while there
 * are at most num_beams of them), then the winners' prefixes and residuals.
 *   X [bs,d]; labels [bs, num_beams, M] int32 out; scores [bs, num_beams] fp32 out (descending wherever a
 *   top-k was taken).  Candidates with equal fp32 score are ordered by ascending (beam, k) index
 *   (torch.topk leaves that order unspecified).                                                            */
int mevi_rq_beam_search(mevi_ctx* ctx, const float* X, int64_t bs, int d, const float* codebook, int M, int K,
                        int metric, int num_beams, int prod, int32_t* labels, float* scores, void* stream);

/* ---- inverted lists ------------------------------------------------------ *
 * replaces: MEVI/pq.py:236-242 / 200-214 (python dict build) with a device
 * sort by leaf key.  key(row) = sum_j codes[row,j] * K^(M-1-j)  (K^M < 2^62).
 *   sorted_docids [n] int32 out: row indices ordered by (key, row) — ascending
 *                 doc id inside a leaf, like the reference's append order
 *   sorted_keys   [n] int64 out: the key of each entry of sorted_docids      */
int mevi_build_inverted_lists(mevi_ctx* ctx, const int32_t* codes, int64_t n, int M, int K, int32_t* sorted_docids,
                              int64_t* sorted_keys, void* stream);
/* replaces: `doc_cluster.get(tuple(leaf), None)` of MEVI/main_models.py:3926-3936 for all (query, leaf) pairs at once.
 *   leaves [n_pairs, M] int64 code tuples (the beam search's output); leaf_keys [n_leaves] int64 ascending, the
 *   distinct keys of mevi_build_inverted_lists; leaf_index [n_pairs] int32 out: position of the tuple's key in
 *   leaf_keys, -1 when no document carries it or a code is outside [0, K).                                        */
int mevi_leaf_lookup(mevi_ctx* ctx, const int64_t* leaves, int64_t n_pairs, int M, int K, const int64_t* leaf_keys,
                     int64_t n_leaves, int32_t* leaf_index, void* stream);
/* Occurrence table of inverted lists in which a document may be listed under several leaves (`--doc_multiclus > 1`):
 * a device sort of (document, CSR position), grouped by document.  *max_occ_host = C, the largest number of positions
 * of any document (0 when n == 0).  With occ_leaves != NULL ([n, width] int32, width >= C - 1) row p receives the CSR
 * leaf indices of the other positions of the document at position p, in ascending position order, -1 padded; a
 * position p' < p in the same leaf (a leaf listing the document twice) is written as -2 - leaf.
 * Synchronises `stream`.  MEVI_ERR_INVALID when width < C - 1.                                                     */
int mevi_occurrence_table(mevi_ctx* ctx, const int64_t* leaf_offsets, int64_t n_leaves, const int32_t* leaf_docids,
                          int64_t n, int width, int32_t* occ_leaves, int32_t* max_occ_host, void* stream);

/* ---- cluster-restricted re-rank ----------------------------------------- *
 * replaces: MEVI/main_models.py:3915-4014 (per query: leaves -> candidate rows
 * -> q.P^T (document_encoder.py:128-132) -> descending sort) for all queries in
 * one call, keeping the k best.
 *   Q [nq,d], D [n,d]
 *   d_layout     0: row i of D is document row i (candidates are gathered row by row)
 *                1: D is stored in CSR order, row j of D is document leaf_docids[j] (see
 *                   mevi_gather_rows) — every leaf is one contiguous byte range, streamed with bulk
 *                   async copies; this is the fast path
 *   leaf_offsets [n_leaves+1] int64 CSR into leaf_docids; leaf_docids int32 document rows
 *   query_leaves [nq,L] int32 CSR leaf index per beam-search leaf, -1 = leaf
 *                holds no document (main_models.py:3928,3935)
 *   scores [nq,k] fp32 out, descending, -inf padded; ids [nq,k] int64 out
 *                (= id_base + row), -1 padded; n_candidates [nq] int32 out
 * Ties between equal scores are ordered by ascending id.                      */
int mevi_cluster_rerank(mevi_ctx* ctx, const float* Q, int nq, const float* D, int64_t n, int d, int d_layout,
                        const int64_t* leaf_offsets, int64_t n_leaves, const int32_t* leaf_docids,
                        const int32_t* query_leaves, int L, int k, int64_t id_base, float* scores, int64_t* ids,
                        int32_t* n_candidates, void* stream);

/* mevi_cluster_rerank restricted to the first max_rows candidate rows of every query (leaf-ordered layout, ids =
 * rows of D_leaf): the exact top-k of a prefix of the candidates.  Its k-th score is a lower bound of the query's
 * final k-th score - the starting threshold of the grouped re-rank below.                                         */
int mevi_cluster_rerank_prefix(mevi_ctx* ctx, const float* Q, int nq, const float* D_leaf, int64_t n, int d,
                               const int64_t* leaf_offsets, int64_t n_leaves, const int32_t* leaf_docids,
                               const int32_t* query_leaves, int L, int k, int64_t max_rows, float* scores, int64_t* ids,
                               int32_t* n_candidates, void* stream);

/* mevi_cluster_rerank (leaf-ordered layout) for an index built with `--doc_multiclus > 1`, where a document is listed
 * under up to C leaves: one entry per document, like main_models.py:3998-4011 followed by the sort and the
 * `[:save_hard_neg]` truncation.  For a query and a document, let c be the number of positions of the query's leaf list
 * whose leaf lists the document (a leaf repeated in the list counts once per position, a leaf listing the document
 * twice counts twice: the reference's concatenation) and s its fp32 score (the same
 * at every position).  Its score is s for aggr = MEVI_MULTICLUS_MAX, and the fp32 fold ((0 + s) + s) + ... of c terms
 * for MEVI_MULTICLUS_ADD.  Output as mevi_cluster_rerank: the k best distinct documents by (score desc, id asc);
 * n_candidates counts occurrences (the reference's cur_ndoc).
 *   occ_leaves [n, C-1] int32 from mevi_occurrence_table (NULL when C == 1): per CSR position, the CSR leaf indices of
 *              the document's other positions, -1 padded.  16-byte aligned; the kernel copies it in 16-byte
 *              aligned pieces, so the allocation must extend to the next multiple of 16 bytes past n*(C-1)*4.
 * MEVI_ERR_UNSUPPORTED for C > 16, and for shapes the streaming kernel does not take.                              */
#define MEVI_MULTICLUS_ADD 0
#define MEVI_MULTICLUS_MAX 1
int mevi_cluster_rerank_multiclus(mevi_ctx* ctx, const float* Q, int nq, const float* D_leaf, int64_t n, int d,
                                  const int64_t* leaf_offsets, int64_t n_leaves, const int32_t* leaf_docids,
                                  const int32_t* occ_leaves, int C, const int32_t* query_leaves, int L, int k, int aggr,
                                  int64_t id_base, float* scores, int64_t* ids, int32_t* n_candidates, void* stream);

/* The same loop keeping EVERY candidate (the shipped recipe runs `--save_hard_neg 8841823`: main_models.py:4012-4014,
 * 4046-4053 write all candidates, sorted): leaf-ordered layout only.  Candidate number pos of query q, in the
 * reference's concatenation order (leaf order = beam order, then row order inside the leaf, 3994-3997), goes to
 * scores/ids[out_offsets[q] + pos]; out_offsets [nq+1] int64 (device) = exclusive prefix sum of the queries' candidate
 * counts, computed by the caller from leaf_offsets and query_leaves.  Sorting (and the doc_multiclus aggregation of
 * 3998-4011) is the caller's: a segmented device sort in mevi_b200/rerank.py.                                      */
int mevi_cluster_rerank_all(mevi_ctx* ctx, const float* Q, int nq, const float* D_leaf, int64_t n, int d,
                            const int64_t* leaf_offsets, int64_t n_leaves, const int32_t* leaf_docids,
                            const int32_t* query_leaves, int L, int64_t id_base, const int64_t* out_offsets, float* scores,
                            int64_t* ids, int32_t* n_candidates, void* stream);

/* The same call, same arguments, same outputs byte for byte (scores, ids, n_candidates), with every leaf's rows read
 * once for all the queries that chose it: work items of one tile of <= 128 rows of a leaf x up to 256 of the leaf's
 * (query, position) pairs, planned on the device inside the call (one host synchronisation).  The fp32 scores follow
 * the streaming kernel's summation order exactly (the lane partials and its shuffle tree, evaluated as a pairwise
 * sum in bit-reversed lane order), so no fp16 image is needed.  Scratch: about 28 bytes per (query, position) pair
 * plus 24 bytes per leaf.                                                                                           */
int mevi_cluster_rerank_all_grouped(mevi_ctx* ctx, const float* Q, int nq, const float* D_leaf, int64_t n, int d,
                                    const int64_t* leaf_offsets, int64_t n_leaves, const int32_t* leaf_docids,
                                    const int32_t* query_leaves, int L, int64_t id_base, const int64_t* out_offsets,
                                    float* scores, int64_t* ids, int32_t* n_candidates, void* stream);

/* Sorts every query's segment [offsets[q], offsets[q+1]) of (scores, ids) by score descending, then id ascending:
 * -0.0 and +0.0 compare equal, NaN comes first, every element keeps its score bits.  This is the order of three stable
 * torch.argsort passes (id, score descending, query) on the device.  offsets [nq+1] int64 device; the outputs may be
 * the inputs.  Every id must lie in [0, 2^32) (MEVI_ERR_INVALID otherwise) and no query may hold 2^31 candidates or
 * more.  Whole queries are sorted in chunks of at most 2^28 candidates (or one larger query), so totals above 2^31
 * work.  Extra device memory: 24 bytes per candidate of the largest chunk (at most 6 GiB below 2^28) plus cub's
 * temporary storage, kept in the context's scratch.  Two host synchronisations (offsets, id check).              */
int mevi_sort_candidates(mevi_ctx* ctx, int nq, const int64_t* offsets, const float* scores_in, const int64_t* ids_in,
                         float* scores_out, int64_t* ids_out, void* stream);

/* ---- cluster-restricted re-rank as leaf-grouped GEMMs (tensor cores) ------ *
 * replaces: the same loop, MEVI/main_models.py:3915-4014.  A leaf selected by many queries is read ONCE and
 * scored against all of them: per leaf a [documents of the leaf] x [queries that chose it] fp16 tcgen05 GEMM whose
 * scores are a prefilter with a rigorous margin; survivors are re-scored in exact fp32 (same contract as the flat
 * search).  Index side, once: tiles of 128 rows of D_leaf that never straddle a leaf
 *   src_index [n_tiles*128] int32   row of D_leaf per image row, -1 = padding
 *   Aimg      [n_tiles][d/64][128][64] fp16 (n_tiles*128*d*2 bytes, caller-owned)
 *   absmax_out, maxnorm_out (host)  scale source and largest document norm; absmax_out < 0: the image cannot
 *                                   carry the guarantee (fp16 range), keep mevi_cluster_rerank.
 * Call side: _begin (query scale, margins, thresholds from tau0 [nq] device or NULL), one _round per batch of
 * (leaf, query) pairs, _finish.  A round takes
 *   tile_row0, tile_nrows [n_tiles] int32; item_tile, item_group [n_items] int32 work items: a document tile meets
 *   up to max_groups_per_item (1, 2 or 4) CONSECUTIVE query groups - item_group = first group | (number of groups << 24),
 *   0 in the high bits = 1 - so that the tile is fetched once for up to 256 queries;
 *   group_qid [n_groups*64] int32 query index per column of a group, -1 = padding.
 * _plan / _plan_fill: the rounds of a call planned on the device (replaces the torch index arithmetic of
 *   mevi_b200/rerank.py plan_grouped_tile_rounds).  ql [nq,L] int32 = leaf index per (query, leaf rank), -1 = none;
 *   leaf_offsets / leaf_tile0 [n_leaves+1] int64 = first row / first tile of every leaf; boot_leaves [n_boot] ascending
 *   leaf-rank boundaries: round i < n_boot = first tile of the leaves with rank in [boot[i-1], boot[i]) (threshold
 *   samples, items of max_groups_sample groups), round n_boot = the remaining first tiles + every further tile of every
 *   leaf against all the queries that chose it (items of max_groups_last groups).  Outputs: ncand [nq] int32 (device)
 *   candidates per query, weak [nq] int32 (device) 1 = the query's sample is too small for its candidate count (fewer rows
 *   than min(boot_min_rows, max(2k, candidates * k / pass_budget)) with more than pass_budget candidates (6,144 of the 8,192
 *   buffer slots is the caller's default): the k-th best of the sample
 *   would let more through the last round than the candidate buffer holds; the caller supplies such a query's tau0 from
 *   mevi_cluster_rerank_prefix), sizes_host [2*(n_boot+1)+1] = (items, groups) per round,
 *   then the number of weak queries.  _plan_fill writes round `round` into caller-allocated item_tile / item_group
 *   [items] and group_qid [groups*64]; ql, leaf_offsets and leaf_tile0 must stay valid until the last _plan_fill.
 * _finish: scores [nq,k] fp32 descending, rows [nq,k] int64 rows of D_leaf, -1 padded; *n_failed = number of queries
 * whose guarantee could not be established (candidate buffer / margin window overflow; marked in failed_or_null [nq]
 * int32 device) - the caller re-runs just those through mevi_cluster_rerank; *n_failed = nq: the whole call is invalid.
 * Thresholds: tau0 (a lower bound of every query's k-th best score) or NULL; with NULL the FIRST round must be small
 * enough that all its scores fit the 8,192-slot candidate buffers (they are all appended), which bootstraps them.
 * The state between _begin and _finish lives in the context: one grouped call at a time per context.            */
int mevi_rerank_grouped_image(mevi_ctx* ctx, const float* D_leaf, int64_t n, int d, const int32_t* src_index,
                              int64_t n_tiles, void* Aimg, float* absmax_out, float* maxnorm_out, void* stream);
int mevi_rerank_grouped_begin(mevi_ctx* ctx, const float* Q, int nq, int d, float d_absmax, float d_maxnorm,
                              const float* tau0, void* stream);
int mevi_rerank_grouped_round(mevi_ctx* ctx, const float* Q, int nq, int d, const void* Aimg, const int32_t* tile_row0,
                              const int32_t* tile_nrows, const int32_t* item_tile, const int32_t* item_group,
                              int64_t n_items, const int32_t* group_qid, int64_t n_groups, int max_groups_per_item,
                              int k, void* stream);
int mevi_rerank_grouped_plan(mevi_ctx* ctx, const int32_t* ql, int nq, int L, const int64_t* leaf_offsets,
                             const int64_t* leaf_tile0, int64_t n_leaves, const int32_t* boot_leaves, int n_boot,
                             int boot_min_rows, int k, int pass_budget, int max_groups_sample, int max_groups_last, int32_t* ncand,
                             int32_t* weak, int64_t* sizes_host, void* stream);
int mevi_rerank_grouped_plan_fill(mevi_ctx* ctx, int round, int32_t* item_tile, int32_t* item_group, int32_t* group_qid,
                                  void* stream);
/* between rounds (and before _finish): raise == 0 copies the call's thresholds [nq] out, raise != 0 lifts them to
 * max(own, tau).  Sharded documents: all-reduce(MAX) in between - the largest local k-th best score is a lower bound of
 * the global one - so every rank filters and re-scores against the global bound.                                    */
int mevi_rerank_grouped_thresholds(mevi_ctx* ctx, int nq, int d, float* tau, int raise, void* stream);
int mevi_rerank_grouped_finish(mevi_ctx* ctx, const float* Q, int nq, const float* D_leaf, int d, int k, float* scores,
                               int64_t* rows, int32_t* failed_or_null, int* n_failed, void* stream);
/* The same call on a multi-cluster index (`--doc_multiclus > 1`): the result of mevi_cluster_rerank_multiclus, bit for
 * bit.  After _begin (tau0 = NULL), _multiclus attaches the index's multi-cluster data to the call:
 *   query_leaves [nq,L] int32 the query's CSR leaves as given (a repeated leaf included: c counts every position),
 *   occ_leaves / C from mevi_occurrence_table (NULL when C == 1), tile_leaf [n_tiles] int32 leaf of every image tile,
 *   aggr MEVI_MULTICLUS_ADD / _MAX.
 * It writes query_leaves_masked [nq,L] int32 (every later position of a repeated leaf and every empty leaf set to -1:
 * the list to plan the rounds with, one pair per distinct leaf) and n_candidates [nq] int32 (occurrences, the
 * reference's cur_ndoc).  The rounds then keep one entry per (query, document), scored by its aggregated approximate
 * score, against a margin widened for the aggregation (DESIGN §4).  The thresholds of mevi_cluster_rerank_prefix
 * are not lower bounds here: a query without a usable threshold sample is given tau = +inf (_thresholds, raise != 0)
 * and re-run by the caller through mevi_cluster_rerank_multiclus.  _finish_multiclus: scores [nq,k] fp32 and
 * ids [nq,k] int64 = id_base + leaf_docids[row], ordered by (aggregated score desc, id asc), -1 padded; failed / n_failed
 * as _finish.  query_leaves, leaf_offsets, occ_leaves and tile_leaf must stay valid until _finish_multiclus.
 * MEVI_ERR_UNSUPPORTED for C > 16 or L > 4096.                                                                      */
int mevi_rerank_grouped_multiclus(mevi_ctx* ctx, int nq, int d, const int32_t* query_leaves, int L,
                                  const int64_t* leaf_offsets, int64_t n_leaves, const int32_t* occ_leaves, int C,
                                  const int32_t* tile_leaf, int aggr, int32_t* query_leaves_masked, int32_t* n_candidates,
                                  void* stream);
int mevi_rerank_grouped_finish_multiclus(mevi_ctx* ctx, const float* Q, int nq, const float* D_leaf, int d, int k,
                                         const int32_t* leaf_docids, int64_t id_base, float* scores, int64_t* ids,
                                         int32_t* failed_or_null, int* n_failed, void* stream);

/* out[i,:] = D[rows[i],:] for i < m: builds the leaf-ordered copy of the document matrix
 * (rows = the CSR's leaf_docids).  Replaces the per-leaf memmap fancy-index gather of
 * MEVI/main_models.py:3944 (IndexedData.__getitem__, 1011-1017) with a one-time permutation.  */
int mevi_gather_rows(mevi_ctx* ctx, const float* D, int64_t n, int d, const int32_t* rows, int64_t m, float* out,
                     void* stream);

/* ---- exact flat inner-product search ------------------------------------ *
 * replaces: MEVI/faiss_search.py:13-21 with param='Flat' (faiss IndexFlatIP
 * add + search): scores [nq,k] fp32 descending (-inf padded), ids [nq,k] int64
 * (= id_base + row, -1 padded).                                               */
int mevi_flat_ip_topk(mevi_ctx* ctx, const float* Q, int nq, const float* D, int64_t n, int d, int k,
                      int64_t id_base, int mode, float* scores, int64_t* ids, void* stream);

/* Persistent form of the same search: faiss `index.add(doc)` once, `index.search(query, k)` many times
 * (faiss_search.py:15-20).  _create converts D [n,d] to the fp16 tile image the tensor path reads (n*d*2 bytes, owned
 * by the index) and records its scale / largest norm; _search then only pays for the query image, the GEMM and the
 * exact fp32 re-score.  D stays caller-owned and must outlive the index (re-score and fp32 fall-back read it).
 * k <= 1024 on the tensor path (the reference CLI default is --topk 1000); other shapes run the fp32 kernel.       */
typedef struct mevi_flat_index mevi_flat_index;
int mevi_flat_index_create(mevi_ctx* ctx, const float* D, int64_t n, int d, mevi_flat_index** out, void* stream);
int mevi_flat_index_search(mevi_ctx* ctx, const mevi_flat_index* index, const float* Q, int nq, int k, int64_t id_base,
                           int mode, float* scores, int64_t* ids, void* stream);
void mevi_flat_index_destroy(mevi_ctx* ctx, mevi_flat_index* index);

/* Merge S per-shard top-k lists (after an all-gather) into one.
 * scores_in [S,nq,k], ids_in [S,nq,k] -> scores/ids [nq,k]; same ordering rule. */
int mevi_topk_merge(mevi_ctx* ctx, const float* scores_in, const int64_t* ids_in, int S, int nq, int k,
                    float* scores, int64_t* ids, void* stream);

/* Merge S per-shard CSRs of rerank_all (after an all-gather) into the whole corpus's: per query, S runs each sorted by
 * (score desc, id asc) -> one run in the same order.  -0.0 and +0.0 compare equal, as the device torch.sort orders
 * them (rerank_all's sort); NaN scores come first.
 *   scores_in / ids_in   the runs, one block per shard: run r of query q is
 *                        [bases[r] + run_offsets[r][q], bases[r] + run_offsets[r][q+1])
 *   bases [S] int64, run_offsets [S][nq+1] int64 (every run_offsets[r] starts at 0 and is non-decreasing)
 *   out_offsets [nq+1] int64 = the per-query sum of the runs' lengths, from 0 to `total`
 *   scratch_scores / scratch_ids [total]: the intermediate result of the ceil(log2 S) two-way merge passes; needed when
 *                        S > 2 (may be NULL otherwise)
 *   scores / ids [total] the merged CSR values.
 * Checks the offsets on the device and synchronises `stream` before merging.  MEVI_ERR_INVALID for S < 1, S > 8 or
 * inconsistent offsets.                                                                                              */
int mevi_merge_sorted_runs(mevi_ctx* ctx, const float* scores_in, const int64_t* ids_in, int S, int nq,
                           const int64_t* bases, const int64_t* run_offsets, const int64_t* out_offsets, int64_t total,
                           float* scratch_scores, int64_t* scratch_ids, float* scores, int64_t* ids, void* stream);

/* ---- dense scorer -------------------------------------------------------- *
 * replaces: MEVI/document_encoder.py:128-132 compute_similarity(bmm=False):
 * out[nq, n] = Q[nq,d] . P[n,d]^T in fp32 (exact FMA accumulation).            */
int mevi_dense_scores(mevi_ctx* ctx, const float* Q, int nq, const float* P, int64_t n, int d, float* out,
                      void* stream);

/* ---- ensemble fusion (SURVEY 8f.2) ---------------------------------------- *
 * replaces: MEVI/ensemble_marco.py:181-191, 221-240 and MEVI/ensemble_nqdpr.py:192-202, 232-251 (python dictionaries
 * per query) and the list look-ups of their evaluators (ensemble_marco.py:20-31, ensemble_nqdpr.py:23-33).
 * Candidate lists are dense [nq,P] (P <= 4096) with an optional per-query length cand_count[nq] (NULL = P).
 *
 * mevi_ensemble_cluster_ranks: cranks[q,c] = index of document cand_ids[q,c]'s RQ leaf (codes[doc, 0..M), the
 *   rqmapping) in the query's ordered leaf list query_leaves[q, 0..L, 0..M) (a repeated leaf keeps its last index),
 *   num_leaves[q] (= number of distinct leaves) when it is not there or the id is the -1 padding, -2 when the id is
 *   outside [0, n_docs) (the reference raises KeyError).
 * mevi_ensemble_fuse: score' = score + alpha / (beta * crank + 1), times (1 - gamma * alpha) when crank == num_leaves;
 *   float64, every operation rounded on its own (bit-identical to the python floats); a document listed several times
 *   keeps its first position and its last value; out_ids / out_scores [nq,P] = the documents by descending fused score,
 *   ties in first-position order, padded with -1 / -inf; out_count[nq] = number of distinct documents.
 * mevi_ensemble_positions: positions[q,g] = index of targets[q,g] in ranked[q, 0..ranked_count[q]) or -1.
 * mevi_ensemble_first_hit: first j with query_index[q] in array[offsets[doc] .. offsets[doc+1]), doc = ranked[q,j]; -1
 *   if none (NQ-DPR inverse-answer lists, test_inverse_offsets.bin / test_inverse_array.bin).                        */
int mevi_ensemble_cluster_ranks(mevi_ctx* ctx, const int64_t* cand_ids, const int32_t* cand_count, int nq, int P,
                                const int32_t* codes, int64_t n_docs, int M, const int32_t* query_leaves, int L,
                                int32_t* cranks, int32_t* num_leaves, void* stream);
int mevi_ensemble_fuse(mevi_ctx* ctx, const int64_t* cand_ids, const double* cand_scores, const int32_t* cranks,
                       const int32_t* cand_count, int nq, int P, double alpha, double beta, double gamma,
                       int num_leaves, int64_t* out_ids, double* out_scores, int32_t* out_count, void* stream);
int mevi_ensemble_positions(mevi_ctx* ctx, const int64_t* ranked, const int32_t* ranked_count, int nq, int P,
                            const int64_t* targets, const int32_t* target_count, int G, int32_t* positions,
                            void* stream);
int mevi_ensemble_first_hit(mevi_ctx* ctx, const int64_t* ranked, const int32_t* ranked_count, int nq, int P,
                            const int64_t* query_index, const int32_t* offsets, int64_t n_offsets,
                            const int32_t* array, int32_t* first_hit, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MEVI_B200_H */
