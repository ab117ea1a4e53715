// merge.cu — segmented merge of S <= 8 sorted runs per query (the cross-rank merge of a sharded rerank_all).
//
// Every rank of a doc-sharded `rerank_all` returns a CSR over the queries whose segments are sorted by (score desc,
// id asc).  After an all-gather the runs sit one block per rank: run r of query q is
// in[bases[r] + run_offsets[r][q] .. bases[r] + run_offsets[r][q+1]).  The merged CSR is out_offsets.
//
// The merge is a tree of ceil(log2 S) two-way merge-path passes (at least one: S = 1 is a copy into the query-major
// layout).  Pass p merges, per query, groups of 2^p runs pairwise; its output keeps the query-major layout of the
// final result: the merged group of runs [r0, r1) of query q sits at out_offsets[q] + (rows of runs < r0 of q).
// Each CTA owns one TILE of consecutive output positions of a pass.  Because the output of every pass tiles [0, total)
// in (query, group) order, a CTA walks the (query, group) jobs its tile intersects; for each it finds the split of its
// two output diagonals with one binary search each (merge path, global memory), loads the A and B pieces into shared
// memory with coalesced loads, merges VT outputs per thread from a merge-path split in shared memory, and stores the
// tile coalesced.  Roofline: HBM — 12 bytes read and 12 written per element per pass.
//
// Order: score descending, then id ascending.  -0.0 and +0.0 compare equal, as the device torch.sort that sorts each
// rank's run orders them (cub's radix sort folds -0.0 onto +0.0); NaN scores come first.  Elements equal in both keys
// (a document listed twice by one query's leaf list) are indistinguishable, so the output does not depend on which run
// gives first.
#include "common.cuh"

namespace {

constexpr int MG_THREADS = 256;
constexpr int MG_VT = 8;                          // outputs per thread
constexpr int MG_TILE = MG_THREADS * MG_VT;       // outputs per CTA
constexpr int MG_MAX_RUNS = 8;

// fp32 -> order-preserving uint32 (larger key = earlier in the output): -0.0 folds onto +0.0, every NaN onto the top
__device__ __forceinline__ uint32_t mg_key(float f) {
  uint32_t u = __float_as_uint(f);
  if (u == 0x80000000u) u = 0u;
  if ((u & 0x7fffffffu) > 0x7f800000u) return 0xffffffffu;
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// strict "x comes before y"
__device__ __forceinline__ bool mg_before(float sx, int64_t ix, float sy, int64_t iy) {
  const uint32_t kx = mg_key(sx), ky = mg_key(sy);
  return kx > ky || (kx == ky && ix < iy);
}

struct MergePass {
  const float* src_s;
  const int64_t* src_i;
  float* dst_s;
  int64_t* dst_i;
  const int64_t* bases;        // gathered layout (first pass) only
  const int64_t* run_offsets;  // [S][nq+1]
  const int64_t* out_offsets;  // [nq+1]
  int64_t total;
  int nq, S, width;            // width = runs per group already merged (1, 2, 4)
  int gathered;                // 1: src is the all-gathered rank-major layout; 0: the query-major layout of a pass
};

__device__ __forceinline__ int64_t run_len(const MergePass& p, int r, int q) {
  const int64_t* o = p.run_offsets + (int64_t)r * (p.nq + 1);
  return o[q + 1] - o[q];
}

// source position of run r of query q; rows_before = rows of the runs < r of query q
__device__ __forceinline__ int64_t run_src(const MergePass& p, int r, int q, int64_t rows_before) {
  if (p.gathered) return p.bases[r] + p.run_offsets[(int64_t)r * (p.nq + 1) + q];
  return p.out_offsets[q] + rows_before;
}

// merge path: number of A elements among the first `diag` outputs of merge(A, B) (A first on equal keys)
__device__ __forceinline__ int64_t merge_path_global(const float* as, const int64_t* ai, int64_t na, const float* bs,
                                                     const int64_t* bi, int64_t nb, int64_t diag) {
  int64_t lo = diag > nb ? diag - nb : 0, hi = diag < na ? diag : na;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    const int64_t j = diag - 1 - mid;
    if (mg_before(bs[j], bi[j], as[mid], ai[mid])) hi = mid;
    else lo = mid + 1;
  }
  return lo;
}

__global__ void __launch_bounds__(MG_THREADS) merge_pass_kernel(MergePass p) {
  __shared__ float s_s[MG_TILE];
  __shared__ int64_t s_i[MG_TILE];
  __shared__ int64_t s_split[2];
  const int64_t tile_beg = (int64_t)blockIdx.x * MG_TILE;
  if (tile_beg >= p.total) return;
  const int64_t tile_end = min(tile_beg + (int64_t)MG_TILE, p.total);
  // query holding tile_beg: the last q with out_offsets[q] <= tile_beg (queries may be empty)
  int lo = 0, hi = p.nq;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (p.out_offsets[mid] <= tile_beg) lo = mid;
    else hi = mid;
  }
  int q = lo;
  int64_t pos = tile_beg;
  while (pos < tile_end) {
    const int64_t qbeg = p.out_offsets[q], qend = p.out_offsets[q + 1];
    if (pos >= qend) {
      ++q;
      continue;
    }
    // the group [r0, r2) of query q holding pos: A = runs [r0, r1), B = runs [r1, r2)
    int64_t before = 0, job_beg = qbeg, a_len = 0, b_len = 0, a_before = 0, b_before = 0;
    int r0 = 0, r1 = 0;
    for (r0 = 0; r0 < p.S; r0 += 2 * p.width) {
      r1 = min(r0 + p.width, p.S);
      const int r2 = min(r0 + 2 * p.width, p.S);
      a_len = 0;
      b_len = 0;
      for (int r = r0; r < r1; ++r) a_len += run_len(p, r, q);
      for (int r = r1; r < r2; ++r) b_len += run_len(p, r, q);
      if (pos < qbeg + before + a_len + b_len) break;
      before += a_len + b_len;
    }
    a_before = before;
    b_before = before + a_len;
    job_beg = qbeg + before;
    const float* as = p.src_s + run_src(p, r0, q, a_before);
    const int64_t* ai = p.src_i + run_src(p, r0, q, a_before);
    const float* bs = p.src_s + (r1 < p.S ? run_src(p, r1, q, b_before) : 0);
    const int64_t* bi = p.src_i + (r1 < p.S ? run_src(p, r1, q, b_before) : 0);
    const int64_t seg_end = min(job_beg + a_len + b_len, tile_end);
    const int64_t d0 = pos - job_beg, d1 = seg_end - job_beg;
    if (threadIdx.x == 0) s_split[0] = merge_path_global(as, ai, a_len, bs, bi, b_len, d0);
    if (threadIdx.x == 32) s_split[1] = merge_path_global(as, ai, a_len, bs, bi, b_len, d1);
    __syncthreads();
    const int64_t a0 = s_split[0], a1 = s_split[1];
    const int64_t b0 = d0 - a0;
    const int na = (int)(a1 - a0), n = (int)(d1 - d0);
    for (int t = threadIdx.x; t < n; t += MG_THREADS) {
      if (t < na) {
        s_s[t] = as[a0 + t];
        s_i[t] = ai[a0 + t];
      } else {
        s_s[t] = bs[b0 + t - na];
        s_i[t] = bi[b0 + t - na];
      }
    }
    __syncthreads();
    // this thread's outputs [diag, diag + VT) of the n: merge path in shared memory, then a serial merge
    const int nb = n - na;
    const int diag = min(threadIdx.x * MG_VT, n);
    int l = diag > nb ? diag - nb : 0, h = diag < na ? diag : na;
    while (l < h) {
      const int mid = (l + h) >> 1;
      const int j = na + diag - 1 - mid;
      if (mg_before(s_s[j], s_i[j], s_s[mid], s_i[mid])) h = mid;
      else l = mid + 1;
    }
    int ia = l, ib = na + diag - l;
    float vs[MG_VT];
    int64_t vi[MG_VT];
#pragma unroll
    for (int v = 0; v < MG_VT; ++v) {
      const bool take_b = ia >= na || (ib < n && mg_before(s_s[ib], s_i[ib], s_s[ia], s_i[ia]));
      const int src = take_b ? ib : ia;
      vs[v] = s_s[src < n ? src : 0];
      vi[v] = s_i[src < n ? src : 0];
      if (take_b) ++ib;
      else ++ia;
    }
    __syncthreads();
#pragma unroll
    for (int v = 0; v < MG_VT; ++v) {
      if (diag + v < n) {
        s_s[diag + v] = vs[v];
        s_i[diag + v] = vi[v];
      }
    }
    __syncthreads();
    for (int t = threadIdx.x; t < n; t += MG_THREADS) {
      p.dst_s[pos + t] = s_s[t];
      p.dst_i[pos + t] = s_i[t];
    }
    __syncthreads();  // shared memory and s_split are reused by the next job of the tile
    pos = seg_end;
  }
}

// One thread per query: every run's segment is non-negative, runs start at 0 and the output segment holds their sum.
__global__ void merge_check_kernel(const int64_t* __restrict__ run_offsets, const int64_t* __restrict__ out_offsets, int S,
                                   int nq, int64_t total, int* __restrict__ bad) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q > nq) return;
  if (q == nq) {
    bool ok = out_offsets[0] == 0 && out_offsets[nq] == total;
    for (int r = 0; r < S; ++r) ok = ok && run_offsets[(int64_t)r * (nq + 1)] == 0;
    if (!ok) atomicOr(bad, 1);
    return;
  }
  int64_t sum = 0;
  bool ok = true;
  for (int r = 0; r < S; ++r) {
    const int64_t c = run_offsets[(int64_t)r * (nq + 1) + q + 1] - run_offsets[(int64_t)r * (nq + 1) + q];
    ok = ok && c >= 0;
    sum += c;
  }
  if (!ok || out_offsets[q + 1] - out_offsets[q] != sum) atomicOr(bad, 1);
}

}  // namespace

extern "C" int mevi_merge_sorted_runs(mevi_ctx* ctx, const float* scores_in, const int64_t* ids_in, int S, int nq,
                                      const int64_t* bases, const int64_t* run_offsets, const int64_t* out_offsets,
                                      int64_t total, float* scratch_scores, int64_t* scratch_ids, float* scores,
                                      int64_t* ids, void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  MEVI_REQUIRE(ctx, S >= 1 && S <= MG_MAX_RUNS, "merge of %d runs: S must be in [1, %d]", S, MG_MAX_RUNS);
  MEVI_REQUIRE(ctx, nq >= 0 && total >= 0, "bad shape (nq=%d, total=%lld)", nq, (long long)total);
  MEVI_REQUIRE(ctx, bases && run_offsets && out_offsets, "NULL argument");
  MEVI_REQUIRE(ctx, total == 0 || (scores_in && ids_in && scores && ids), "NULL argument");
  MEVI_REQUIRE(ctx, S <= 2 || total == 0 || (scratch_scores && scratch_ids), "a merge of %d runs needs the scratch buffers", S);
  if (int rc = mevi_deferred_error(ctx)) return rc;
  int* d_bad = (int*)mevi_ws(ctx, WS_MISC, 64);
  if (!d_bad) return MEVI_ERR_NOMEM;
  MEVI_CUDA(ctx, cudaMemsetAsync(d_bad, 0, sizeof(int), st));
  merge_check_kernel<<<(unsigned)((nq + 1 + 255) / 256), 256, 0, st>>>(run_offsets, out_offsets, S, nq, total, d_bad);
  MEVI_COUNT_LAUNCH(ctx, 1);
  MEVI_CUDA(ctx, cudaGetLastError());
  int h_bad = 0;
  MEVI_CUDA(ctx, cudaMemcpyAsync(&h_bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, st));
  MEVI_CUDA(ctx, cudaStreamSynchronize(st));
  MEVI_REQUIRE(ctx, h_bad == 0, "inconsistent offsets: every run must start at 0 and grow, and out_offsets must be their "
                                "per-query sum, from 0 to total = %lld", (long long)total);
  if (total == 0) return MEVI_OK;
  int n_pass = 1;
  while ((1 << n_pass) < S) ++n_pass;
  const int64_t grid = (total + MG_TILE - 1) / MG_TILE;
  MEVI_REQUIRE(ctx, grid < (int64_t)2147483647, "total too large");
  // the last pass writes the caller's output: ping-pong backwards from it
  const float* src_s = scores_in;
  const int64_t* src_i = ids_in;
  for (int pass = 0; pass < n_pass; ++pass) {
    const bool to_out = ((n_pass - 1 - pass) & 1) == 0;
    MergePass p;
    p.src_s = src_s;
    p.src_i = src_i;
    p.dst_s = to_out ? scores : scratch_scores;
    p.dst_i = to_out ? ids : scratch_ids;
    p.bases = bases;
    p.run_offsets = run_offsets;
    p.out_offsets = out_offsets;
    p.total = total;
    p.nq = nq;
    p.S = S;
    p.width = 1 << pass;
    p.gathered = pass == 0;
    merge_pass_kernel<<<(unsigned)grid, MG_THREADS, 0, st>>>(p);
    MEVI_COUNT_LAUNCH(ctx, 1);
    MEVI_CUDA(ctx, cudaGetLastError());
    src_s = p.dst_s;
    src_i = p.dst_i;
  }
  return MEVI_OK;
}
