// rerank_all.cu — every candidate of every query: the leaf-grouped fp32 scorer and the per-query device sort.
//
// mevi_cluster_rerank_all_grouped fills the same arrays as mevi_cluster_rerank_all (rerank.cu), byte for byte, but
// reads a leaf's rows once for all the queries that chose it instead of once per query.
//
// The identity.  The streaming kernel gives lane l the partial p_l = fmaf chain, from +0.0f, over t = 0 .. NCH-1 and
// the components x, y, z, w of columns 4(l + 32t) .. 4(l + 32t) + 3 (columns >= d are 0 * 0 terms), then returns
// warp_sum(p): xor shuffles with offsets 16, 8, 4, 2, 1.  fp32 addition is commutative, so every lane ends with the
// same value, a fixed binary tree over p_0 .. p_31 whose leaves, left to right, are the lanes in 5-bit bit-reversed
// order (0, 16, 8, 24, 4, ...).  A thread evaluates it as a running pairwise sum over positions i = 0 .. 31 (slice
// brev5(i)): the partial of position i is added to the pending subtree of level b for every trailing one bit b of i,
// so at most 5 pending partials per (query, row) pair are live.  The result is the streaming kernel's bit for bit,
// including the sign of a zero score.
//
// The schedule.  A work item is one tile of <= 128 rows of one leaf (never straddling leaves) x up to 256 of the pairs
// (query, position in its leaf list) whose leaf it is.  Items are numbered tile-major inside a leaf, so the items of
// one tile run back to back and the tile's second and later reads come from L2.  The CTA stages 32 rows at a time in
// shared memory (whole rows, one coalesced copy; row stride padded so that the 32 lanes' 16-byte loads of one column
// are conflict-free), lane = row.  The pairs are taken 32 at a time: warp w scores RN consecutive pairs, RN = 4, 2 or 1
// as the chunk's width allows, so a thin group (a leaf chosen by a handful of queries, L = 10) spreads over the
// warps instead of filling 64 columns.  Query values are warp-uniform loads (one transaction, L1 / L2: the queries are
// far smaller than L2).  Writes: per pair, 32 consecutive scores and ids.
//
// The plan is made on the device inside the call: pairs counted per leaf with an arrival number (the counting of
// rerank_plan.cu), two exclusive scans (items, pairs), then a counting sort of the pairs by leaf that also stores each
// pair's output base.  One host synchronisation (the number of items, for the grid).
//
// mevi_sort_candidates sorts every query's segment of a CSR by (score desc, id asc) with cub's segmented sort
// on one 64-bit key: the order-preserving image of the score (-0.0 folded onto +0.0, every NaN first) above the
// 32-bit id.  The original score bits ride along as the value, so -0.0 stays -0.0.
#include <cub/cub.cuh>

#include <vector>

#include "common.cuh"

namespace {

constexpr int RA_TILE = 128;       // rows of a leaf tile
constexpr int RA_SUB = 32;         // rows staged in shared memory at a time (one per lane)
constexpr int RA_THREADS = 256;
constexpr int RA_WARPS = RA_THREADS / 32;
constexpr int RA_PASS = RA_WARPS * 4;  // pairs per pass: 8 warps x up to 4 pairs
constexpr int RA_ITEM_COLS = 256;  // pairs per work item

struct AllPlan {
  const int32_t* ql; int nq; int L;
  const int64_t* leaf_offsets; int64_t n_leaves;
  const int64_t* out_offsets;
  int32_t* n_candidates;
  int32_t* cnt;        // [n_leaves + 1] pairs per leaf (+ a trailing 0 for the scan)
  int32_t* arrival;    // [nq * L] arrival number of the pair among its leaf's pairs
  int64_t* items;      // [n_leaves + 1] work items per leaf (+ a trailing 0)
  int64_t* item0;      // exclusive sums of items
  int32_t* pair0;      // exclusive sums of cnt
  int32_t* col_q;      // [pairs] query of the pair, pairs sorted by leaf
  int64_t* col_base;   // [pairs] out_offsets[q] + rows before the pair's position - first row of the leaf
};

// one CTA per query: the pairs' arrival numbers, the query's candidate count, and each pair's output base
__global__ void __launch_bounds__(128) ra_count_kernel(AllPlan p, int64_t* __restrict__ pair_base) {
  using Scan = cub::BlockScan<long long, 128>;
  __shared__ typename Scan::TempStorage tmp;
  __shared__ long long s_carry;
  const int q = blockIdx.x;
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  const int64_t obase = p.out_offsets[q];
  for (int r0 = 0; r0 < p.L; r0 += 128) {
    const int r = r0 + threadIdx.x;
    const int64_t pair = (int64_t)q * p.L + r;
    int leaf = -1;
    long long size = 0;
    if (r < p.L) {
      leaf = p.ql[pair];
      if (leaf >= 0 && leaf < p.n_leaves) size = p.leaf_offsets[leaf + 1] - p.leaf_offsets[leaf];
    }
    long long before, chunk;
    Scan(tmp).ExclusiveSum(size, before, chunk);
    const long long carry = s_carry;
    if (size > 0) {
      p.arrival[pair] = atomicAdd(&p.cnt[leaf], 1);
      pair_base[pair] = obase + carry + before - p.leaf_offsets[leaf];
    }
    __syncthreads();
    if (threadIdx.x == 0) s_carry = carry + chunk;
    __syncthreads();
  }
  if (threadIdx.x == 0 && p.n_candidates) p.n_candidates[q] = (int32_t)(s_carry > 0x7fffffffll ? 0x7fffffffll : s_carry);
}

__global__ void ra_leaf_kernel(AllPlan p) {
  const int64_t leaf = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (leaf > p.n_leaves) return;
  if (leaf == p.n_leaves) {
    p.items[leaf] = 0;
    p.cnt[leaf] = 0;
    return;
  }
  const int64_t rows = p.leaf_offsets[leaf + 1] - p.leaf_offsets[leaf];
  const int64_t tiles = (rows + RA_TILE - 1) / RA_TILE;
  const int c = p.cnt[leaf];
  p.items[leaf] = c > 0 ? tiles * ((c + RA_ITEM_COLS - 1) / RA_ITEM_COLS) : 0;
}

__global__ void ra_fill_kernel(AllPlan p, const int64_t* __restrict__ pair_base) {
  const int64_t pair = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (pair >= (int64_t)p.nq * p.L) return;
  const int leaf = p.ql[pair];
  if (leaf < 0 || leaf >= p.n_leaves || p.leaf_offsets[leaf + 1] == p.leaf_offsets[leaf]) return;
  const int64_t col = (int64_t)p.pair0[leaf] + p.arrival[pair];
  p.col_q[col] = (int32_t)(pair / p.L);
  p.col_base[col] = pair_base[pair];
}

struct ScoreParams {
  const float* Q; const float* D; int d; int stride;
  const int64_t* leaf_offsets; int64_t n_leaves;
  const int32_t* leaf_docids; int64_t id_base;
  const int64_t* item0; const int32_t* cnt; const int32_t* pair0;
  const int32_t* col_q; const int64_t* col_base;
  float* scores; int64_t* ids;
};

// Position i of the tree: v (its slice's partial) absorbs the pending subtree of level B while bit B of i is one; the
// first zero bit parks the result as the pending subtree of that level.  i is warp-uniform, so are the branches.
template <int B, int RN>
__device__ __forceinline__ void ra_combine(int i, float (&st)[5][RN], float (&v)[RN]) {
  if ((i >> B) & 1) {
#pragma unroll
    for (int j = 0; j < RN; ++j) v[j] = st[B][j] + v[j];
    if constexpr (B < 4) ra_combine<B + 1, RN>(i, st, v);
  } else {
#pragma unroll
    for (int j = 0; j < RN; ++j) st[B][j] = v[j];
  }
}

// Scores of this lane's row (s_row) against RN queries: the dense scorer's lane partials, combined in its tree.
template <int NCH, int RN>
__device__ __forceinline__ void ra_score(const ScoreParams& p, const float* s_row, const int32_t* qid, float* out) {
  int qoff[RN];  // nq * d < 2^31 (checked by the caller)
#pragma unroll
  for (int j = 0; j < RN; ++j) qoff[j] = (qid[j] < 0 ? 0 : qid[j]) * p.d;
  float st[5][RN];
  float v[RN];
#pragma unroll 1
  for (int i = 0; i < 32; ++i) {
    const int l = (int)(__brev((unsigned)i) >> 27);
#pragma unroll
    for (int j = 0; j < RN; ++j) v[j] = 0.f;
#pragma unroll
    for (int t = 0; t < NCH; ++t) {
      const int c4 = 4 * (l + 32 * t);
      float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
      float4 qv[RN];
#pragma unroll
      for (int j = 0; j < RN; ++j) qv[j] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c4 < p.d) {  // warp-uniform
        r = *reinterpret_cast<const float4*>(s_row + c4);
#pragma unroll
        for (int j = 0; j < RN; ++j) qv[j] = ldg_f4(p.Q + (qoff[j] + c4));
      }
#pragma unroll
      for (int j = 0; j < RN; ++j) {
        v[j] = fmaf(qv[j].x, r.x, v[j]);
        v[j] = fmaf(qv[j].y, r.y, v[j]);
        v[j] = fmaf(qv[j].z, r.z, v[j]);
        v[j] = fmaf(qv[j].w, r.w, v[j]);
      }
    }
    ra_combine<0, RN>(i, st, v);  // position i closes the pending subtrees of its trailing one bits
  }
#pragma unroll
  for (int j = 0; j < RN; ++j) out[j] = v[j];  // i = 31: the whole tree
}

template <int NCH, int RN>
__device__ __forceinline__ void ra_pairs(const ScoreParams& p, const float* s_row, int64_t c, int n, int64_t row,
                                         bool row_ok, int64_t id) {
  int32_t qid[RN];
#pragma unroll
  for (int j = 0; j < RN; ++j) qid[j] = j < n ? p.col_q[c + j] : -1;
  float s[RN];
  ra_score<NCH, RN>(p, s_row, qid, s);
  if (!row_ok) return;
#pragma unroll
  for (int j = 0; j < RN; ++j) {
    if (j < n) {
      const int64_t o = p.col_base[c + j] + row;
      p.scores[o] = s[j];
      p.ids[o] = id;
    }
  }
}

// two CTAs per SM up to d = 768 (2 x 99 KB of staged rows); d > 768 stages 131 KB, one CTA
template <int NCH>
__global__ void __launch_bounds__(RA_THREADS, NCH > 6 ? 1 : 2) rerank_all_grouped_kernel(ScoreParams p) {
  extern __shared__ __align__(16) float s_rows[];  // [RA_SUB][stride]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t item = blockIdx.x;
  int64_t lo = 0, hi = p.n_leaves;  // the leaf: last with item0[leaf] <= item
  while (hi - lo > 1) {
    const int64_t mid = (lo + hi) >> 1;
    if (p.item0[mid] <= item) lo = mid; else hi = mid;
  }
  const int64_t leaf = lo;
  const int npairs = p.cnt[leaf];
  const int chunks = (npairs + RA_ITEM_COLS - 1) / RA_ITEM_COLS;
  const int64_t loc = item - p.item0[leaf];
  const int64_t lbeg = p.leaf_offsets[leaf], lend = p.leaf_offsets[leaf + 1];
  const int64_t r0 = lbeg + (loc / chunks) * RA_TILE;
  const int nrows = (int)min((int64_t)RA_TILE, lend - r0);
  const int cc = (int)(loc % chunks);
  const int64_t c0 = (int64_t)p.pair0[leaf] + (int64_t)cc * RA_ITEM_COLS;
  const int ncols = min(RA_ITEM_COLS, npairs - cc * RA_ITEM_COLS);
  const int d4 = p.d >> 2;
  const float* s_row = s_rows + lane * p.stride;
  for (int sub = 0; sub < nrows; sub += RA_SUB) {
    const int nr = min(RA_SUB, nrows - sub);
    const float4* src = reinterpret_cast<const float4*>(p.D + (r0 + sub) * p.d);
    for (int e = threadIdx.x; e < nr * d4; e += RA_THREADS) {
      const int rr = e / d4, c = e - rr * d4;
      *reinterpret_cast<float4*>(s_rows + rr * p.stride + 4 * c) = ld_stream_f4(reinterpret_cast<const float*>(src + e));
    }
    const int64_t row = r0 + sub + lane;
    const bool row_ok = lane < nr;
    const int64_t id = row_ok ? p.id_base + (int64_t)p.leaf_docids[row] : 0;
    __syncthreads();
    for (int pc = 0; pc < ncols; pc += RA_PASS) {
      const int w = min(RA_PASS, ncols - pc);
      const int per = (w + RA_WARPS - 1) / RA_WARPS;  // pairs per warp, rounded up to 1, 2, 4 or 8
      const int rn = per <= 1 ? 1 : per <= 2 ? 2 : 4;
      const int first = warp * rn;
      if (first >= w) continue;
      const int n = min(rn, w - first);
      const int64_t c = c0 + pc + first;
      if (rn == 1) ra_pairs<NCH, 1>(p, s_row, c, n, row, row_ok, id);
      else if (rn == 2) ra_pairs<NCH, 2>(p, s_row, c, n, row, row_ok, id);
      else ra_pairs<NCH, 4>(p, s_row, c, n, row, row_ok, id);
    }
    __syncthreads();  // the staged rows are overwritten by the next 32
  }
}

template <int NCH>
cudaError_t launch_rerank_all_grouped(const ScoreParams& p, int64_t n_items, size_t smem, cudaStream_t st) {
  cudaError_t e = cudaFuncSetAttribute(rerank_all_grouped_kernel<NCH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  rerank_all_grouped_kernel<NCH><<<(unsigned)n_items, RA_THREADS, smem, st>>>(p);
  return cudaGetLastError();
}

size_t ra_layout(AllPlan* p, int64_t n_pairs_max, char* ws, size_t* o_base) {
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = (off + bytes + 255) & ~size_t(255); return o; };
  const int64_t nl1 = p->n_leaves + 1;
  const size_t o_cnt = take(nl1 * 4), o_arr = take(n_pairs_max * 4), o_items = take(nl1 * 8), o_item0 = take(nl1 * 8),
               o_pair0 = take(nl1 * 4), o_q = take(n_pairs_max * 4), o_col = take(n_pairs_max * 8), o_pb = take(n_pairs_max * 8);
  if (ws) {
    p->cnt = (int32_t*)(ws + o_cnt); p->arrival = (int32_t*)(ws + o_arr); p->items = (int64_t*)(ws + o_items);
    p->item0 = (int64_t*)(ws + o_item0); p->pair0 = (int32_t*)(ws + o_pair0); p->col_q = (int32_t*)(ws + o_q);
    p->col_base = (int64_t*)(ws + o_col);
  }
  *o_base = o_pb;
  return off;
}

// ---- the per-query sort -------------------------------------------------------------------------------------------
// fp32 -> order-preserving uint32 (larger = earlier): -0.0 folds onto +0.0, every NaN onto the top (merge.cu's key)
__device__ __forceinline__ uint32_t sc_key(float f) {
  uint32_t u = __float_as_uint(f);
  if (u == 0x80000000u) u = 0u;
  if ((u & 0x7fffffffu) > 0x7f800000u) return 0xffffffffu;
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// ids must lie in [0, 2^32): the key holds 32 bits of the id
__global__ void sc_check_kernel(const int64_t* __restrict__ ids, int64_t n, int* __restrict__ bad) {
  bool b = false;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t v = ids[i];
    b |= v < 0 || v > 0xffffffffll;
  }
  if (__any_sync(MEVI_FULL_MASK, b) && (threadIdx.x & 31) == 0) atomicOr(bad, 1);
}

__global__ void sc_pack_kernel(const float* __restrict__ scores, const int64_t* __restrict__ ids, int64_t n,
                               uint64_t* __restrict__ keys, uint32_t* __restrict__ vals) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float s = scores[i];
    keys[i] = ((uint64_t)(~sc_key(s)) << 32) | (uint64_t)(uint32_t)ids[i];
    vals[i] = __float_as_uint(s);
  }
}

__global__ void sc_unpack_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ vals, int64_t n,
                                 float* __restrict__ scores, int64_t* __restrict__ ids) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    scores[i] = __uint_as_float(vals[i]);
    ids[i] = (int64_t)(keys[i] & 0xffffffffull);
  }
}

__global__ void sc_rel_offsets_kernel(const int64_t* __restrict__ offsets, int q0, int nseg, int* __restrict__ rel) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i <= nseg) rel[i] = (int)(offsets[q0 + i] - offsets[q0]);
}

constexpr int64_t SC_CHUNK = (int64_t)1 << 28;  // items per sort: bounds the workspace (24 bytes per item)

}  // namespace

extern "C" {

int mevi_cluster_rerank_all_grouped(mevi_ctx* ctx, const float* Q, int nq, const float* D_leaf, int64_t n, int d,
                                    const int64_t* leaf_offsets, int64_t n_leaves, const int32_t* leaf_docids,
                                    const int32_t* query_leaves, int L, int64_t id_base, const int64_t* out_offsets,
                                    float* scores, int64_t* ids, int32_t* n_candidates, void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  MEVI_REQUIRE(ctx, Q && D_leaf && leaf_offsets && leaf_docids && query_leaves && out_offsets && scores && ids, "NULL argument");
  MEVI_REQUIRE(ctx, d > 0 && d % 4 == 0 && d <= 1024, "re-rank needs d %% 4 == 0 and d <= 1024 (got %d)", d);
  MEVI_REQUIRE(ctx, L >= 1 && L <= 4096, "L must be in [1, 4096] (got %d)", L);
  MEVI_REQUIRE(ctx, n_leaves >= 0 && n_leaves < (int64_t)1 << 30, "bad n_leaves");
  if (nq <= 0) return MEVI_OK;
  const int64_t n_pairs = (int64_t)nq * L;
  MEVI_REQUIRE(ctx, n_pairs < (int64_t)1 << 31 && (int64_t)nq * d < (int64_t)1 << 31, "nq * L and nq * d must be below 2^31");
  if (int rc = mevi_deferred_error(ctx)) return rc;
  AllPlan p;
  p.ql = query_leaves; p.nq = nq; p.L = L; p.leaf_offsets = leaf_offsets; p.n_leaves = n_leaves;
  p.out_offsets = out_offsets; p.n_candidates = n_candidates;
  size_t o_base = 0;
  const size_t bytes = ra_layout(&p, n_pairs, nullptr, &o_base);
  char* ws = (char*)mevi_ws(ctx, WS_RA_PLAN, bytes);
  if (!ws) return MEVI_ERR_NOMEM;
  ra_layout(&p, n_pairs, ws, &o_base);
  int64_t* pair_base = (int64_t*)(ws + o_base);
  size_t tmp_items = 0, tmp_pairs = 0;
  MEVI_CUDA(ctx, cub::DeviceScan::ExclusiveSum(nullptr, tmp_items, p.items, p.item0, (int)(n_leaves + 1), st));
  MEVI_CUDA(ctx, cub::DeviceScan::ExclusiveSum(nullptr, tmp_pairs, p.cnt, p.pair0, (int)(n_leaves + 1), st));
  const size_t tmp_bytes = tmp_items > tmp_pairs ? tmp_items : tmp_pairs;
  void* tmp = mevi_ws(ctx, WS_SORT_TMP, tmp_bytes);
  if (!tmp) return MEVI_ERR_NOMEM;
  MEVI_CUDA(ctx, cudaMemsetAsync(p.cnt, 0, (size_t)(n_leaves + 1) * 4, st));
  ra_count_kernel<<<nq, 128, 0, st>>>(p, pair_base);
  ra_leaf_kernel<<<(unsigned)((n_leaves + 1 + 255) / 256), 256, 0, st>>>(p);
  size_t tb = tmp_bytes;
  MEVI_CUDA(ctx, cub::DeviceScan::ExclusiveSum(tmp, tb, p.items, p.item0, (int)(n_leaves + 1), st));
  tb = tmp_bytes;
  MEVI_CUDA(ctx, cub::DeviceScan::ExclusiveSum(tmp, tb, p.cnt, p.pair0, (int)(n_leaves + 1), st));
  ra_fill_kernel<<<(unsigned)((n_pairs + 255) / 256), 256, 0, st>>>(p, pair_base);
  MEVI_CUDA(ctx, cudaGetLastError());
  MEVI_COUNT_LAUNCH(ctx, 5);
  int64_t n_items = 0;
  MEVI_CUDA(ctx, cudaMemcpyAsync(&n_items, p.item0 + n_leaves, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  MEVI_CUDA(ctx, cudaStreamSynchronize(st));
  if (n_items == 0) return MEVI_OK;
  MEVI_REQUIRE(ctx, n_items < (int64_t)2147483647, "too many work items (%lld)", (long long)n_items);
  ScoreParams s;
  s.Q = Q; s.D = D_leaf; s.d = d;
  s.stride = ((d / 4) & 1) ? d : d + 4;  // 16-byte row stride odd: a quarter warp's 16-byte loads of one column hit distinct banks
  s.leaf_offsets = leaf_offsets; s.n_leaves = n_leaves; s.leaf_docids = leaf_docids; s.id_base = id_base;
  s.item0 = p.item0; s.cnt = p.cnt; s.pair0 = p.pair0; s.col_q = p.col_q; s.col_base = p.col_base;
  s.scores = scores; s.ids = ids;
  const size_t smem = (size_t)RA_SUB * s.stride * sizeof(float);
  cudaError_t e;
  if (d <= 128) e = launch_rerank_all_grouped<1>(s, n_items, smem, st);
  else if (d <= 256) e = launch_rerank_all_grouped<2>(s, n_items, smem, st);
  else if (d <= 512) e = launch_rerank_all_grouped<4>(s, n_items, smem, st);
  else if (d <= 768) e = launch_rerank_all_grouped<6>(s, n_items, smem, st);
  else e = launch_rerank_all_grouped<8>(s, n_items, smem, st);
  if (e != cudaSuccess) return mevi_set_error(ctx, MEVI_ERR_CUDA, "rerank_all_grouped launch: %s", cudaGetErrorString(e));
  MEVI_COUNT_LAUNCH(ctx, 1);
  return MEVI_OK;
}

int mevi_sort_candidates(mevi_ctx* ctx, int nq, const int64_t* offsets, const float* scores_in, const int64_t* ids_in,
                         float* scores_out, int64_t* ids_out, void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  MEVI_REQUIRE(ctx, nq >= 0 && offsets, "bad argument");
  if (nq == 0) return MEVI_OK;
  if (int rc = mevi_deferred_error(ctx)) return rc;
  std::vector<int64_t> off(nq + 1);
  MEVI_CUDA(ctx, cudaMemcpyAsync(off.data(), offsets, (size_t)(nq + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  MEVI_CUDA(ctx, cudaStreamSynchronize(st));
  bool ok = off[0] == 0;
  for (int q = 0; q < nq && ok; ++q) ok = off[q + 1] >= off[q];
  MEVI_REQUIRE(ctx, ok, "offsets must start at 0 and not decrease");
  const int64_t total = off[nq];
  if (total == 0) return MEVI_OK;
  MEVI_REQUIRE(ctx, scores_in && ids_in && scores_out && ids_out, "NULL argument");
  int* chk = (int*)mevi_ws(ctx, WS_MISC, 64);
  if (!chk) return MEVI_ERR_NOMEM;
  MEVI_CUDA(ctx, cudaMemsetAsync(chk, 0, sizeof(int), st));
  const unsigned grid = (unsigned)(4 * ctx->sm_count);
  sc_check_kernel<<<grid, 256, 0, st>>>(ids_in, total, chk);
  MEVI_CUDA(ctx, cudaGetLastError());
  MEVI_COUNT_LAUNCH(ctx, 1);
  int h_bad = 0;
  MEVI_CUDA(ctx, cudaMemcpyAsync(&h_bad, chk, sizeof(int), cudaMemcpyDeviceToHost, st));
  MEVI_CUDA(ctx, cudaStreamSynchronize(st));
  MEVI_REQUIRE(ctx, h_bad == 0, "sort_candidates: every id must lie in [0, 2^32)");
  // chunks of whole queries, each below SC_CHUNK items unless one query alone is larger (then that query, < 2^31)
  std::vector<int> bounds{0};
  int64_t biggest = 0;
  for (int q = 0; q < nq; ++q) {
    const int64_t seg = off[q + 1] - off[q];
    MEVI_REQUIRE(ctx, seg < (int64_t)2147483647, "a query holds %lld candidates (at most 2^31 - 1)", (long long)seg);
    if (off[q + 1] - off[bounds.back()] > SC_CHUNK && q > bounds.back()) bounds.push_back(q);
  }
  bounds.push_back(nq);
  for (size_t b = 0; b + 1 < bounds.size(); ++b) {
    const int64_t items = off[bounds[b + 1]] - off[bounds[b]];
    biggest = items > biggest ? items : biggest;
  }
  // keys (two buffers), values (two buffers), chunk-relative offsets
  const size_t kb = ((size_t)biggest * 8 + 255) & ~size_t(255), vb = ((size_t)biggest * 4 + 255) & ~size_t(255);
  int max_seg = 0;
  for (size_t b = 0; b + 1 < bounds.size(); ++b) max_seg = max(max_seg, bounds[b + 1] - bounds[b]);
  const size_t ob = ((size_t)(max_seg + 1) * 4 + 255) & ~size_t(255);
  char* ws = (char*)mevi_ws(ctx, WS_RA_SORT, 2 * kb + 2 * vb + ob);
  if (!ws) return MEVI_ERR_NOMEM;
  uint64_t* k0 = (uint64_t*)ws;
  uint64_t* k1 = (uint64_t*)(ws + kb);
  uint32_t* v0 = (uint32_t*)(ws + 2 * kb);
  uint32_t* v1 = (uint32_t*)(ws + 2 * kb + vb);
  int* rel = (int*)(ws + 2 * kb + 2 * vb);
  size_t tmp_bytes = 0;
  {
    cub::DoubleBuffer<uint64_t> dk(k0, k1);
    cub::DoubleBuffer<uint32_t> dv(v0, v1);
    MEVI_CUDA(ctx, cub::DeviceSegmentedSort::SortPairs(nullptr, tmp_bytes, dk, dv, (int)biggest, max_seg, rel, rel + 1, st));
  }
  void* tmp = mevi_ws(ctx, WS_SORT_TMP, tmp_bytes);
  if (!tmp) return MEVI_ERR_NOMEM;
  for (size_t b = 0; b + 1 < bounds.size(); ++b) {
    const int q0 = bounds[b], nseg = bounds[b + 1] - q0;
    const int64_t base = off[q0], items = off[bounds[b + 1]] - base;
    if (items == 0) continue;
    sc_rel_offsets_kernel<<<(nseg + 1 + 255) / 256, 256, 0, st>>>(offsets, q0, nseg, rel);
    sc_pack_kernel<<<grid, 256, 0, st>>>(scores_in + base, ids_in + base, items, k0, v0);
    cub::DoubleBuffer<uint64_t> dk(k0, k1);
    cub::DoubleBuffer<uint32_t> dv(v0, v1);
    size_t tb = tmp_bytes;
    MEVI_CUDA(ctx, cub::DeviceSegmentedSort::SortPairs(tmp, tb, dk, dv, (int)items, nseg, rel, rel + 1, st));
    sc_unpack_kernel<<<grid, 256, 0, st>>>(dk.Current(), dv.Current(), items, scores_out + base, ids_out + base);
    MEVI_CUDA(ctx, cudaGetLastError());
    MEVI_COUNT_LAUNCH(ctx, 3);
  }
  return MEVI_OK;
}

}  // extern "C"
