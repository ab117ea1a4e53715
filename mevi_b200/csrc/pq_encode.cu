// pq_encode.cu — product-quantiser encode (pq_type 'pq' / 'opq' after rotation).
// Replaces MEVI/pq.py:249-279 get_pq_document_cluster: for every row and every sub-vector j the nearest
// centroid of codebook[j] under compute_scores (pq.py:124-131): argmax_k -sum_e (a_e - b_e)^2 ('l2') or
// argmax_k sum_e a_e*b_e ('ip'), lowest index on exact fp32 ties (torch.max semantics).  Direct-form fp32 on
// CUDA cores, the literal restatement of the reference arithmetic (sub-vector widths of 24-192 floats are too
// narrow to amortise an operand conversion, and K*dsub*M = K*d floats of codebook stay L1/L2 resident).
//
// A CTA stages a tile of 32 rows in shared memory (coalesced 128-bit loads, row pitch d+4 floats so the
// per-lane 128-bit reads below are conflict-free); lane = row, each warp takes sub-vectors j = warp, warp+8, ...
// and walks the K centroids of codebook[j] with warp-uniform (broadcast) 128-bit loads.
// Roofline: FP32 issue (3*K*d flops per row against 4*d bytes).  Measured (8,841,823 x 768, bench `widened_rows`).
#include <math_constants.h>
#include <stdlib.h>

#include "common.cuh"

namespace {

constexpr int PQ_THREADS = 256;
constexpr int PQ_ROWS = 32;

template <bool L2>
__global__ void __launch_bounds__(PQ_THREADS) pq_encode_kernel(const float* __restrict__ X, int64_t n, int d,
                                                               const float* __restrict__ cb, int M, int K, int dsub,
                                                               int32_t* __restrict__ codes,
                                                               const int32_t* __restrict__ work_rows,   // optional: row ids
                                                               const int64_t* __restrict__ n_work_dev,  // and their count
                                                               const int* __restrict__ run_if)          // optional: run only if != 0
{
  if (run_if != nullptr && *run_if == 0) return;
  // work-list form (the arbiter of rows the tensor prefilter flagged): item i is row work_rows[i]; the arithmetic per
  // (row, sub-vector, centroid) does not depend on the tile a row sits in, so codes equal those of the plain form
  if (work_rows != nullptr) n = *n_work_dev;
  extern __shared__ __align__(16) float sx[];  // [PQ_ROWS][d + 4]
  const int pitch = d + 4;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int d4 = d >> 2, ds4 = dsub >> 2;
  const int nparts = M >= PQ_THREADS / 32 ? 1 : (PQ_THREADS / 32) / M;
  const int ntasks = M * nparts;
  float* s_bs = sx + PQ_ROWS * pitch;                       // [ntasks][PQ_ROWS] best score of a task
  int* s_bi = reinterpret_cast<int*>(s_bs + ntasks * PQ_ROWS);  // [ntasks][PQ_ROWS] its centroid
  const int64_t n_tiles = (n + PQ_ROWS - 1) / PQ_ROWS;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t r0 = tile * PQ_ROWS;
    const int rows = (int)((n - r0) < PQ_ROWS ? (n - r0) : PQ_ROWS);
    __syncthreads();  // previous tile fully consumed
    for (int i = tid; i < PQ_ROWS * d4; i += PQ_THREADS) {
      const int r = i / d4, c = i - r * d4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < rows) v = ld_stream_f4(X + (work_rows ? (int64_t)work_rows[r0 + r] : r0 + r) * d + 4 * c);
      *reinterpret_cast<float4*>(sx + r * pitch + 4 * c) = v;
    }
    __syncthreads();
    // task = (sub-vector j, slice of the K centroids): with fewer than 8 sub-vectors the K range is cut so that all
    // eight warps work.  Two centroids at a time, four partial sums each: eight independent FMA chains per lane
    // (one serial chain per centroid left the FP32 pipe waiting on its own latency).
    for (int task = warp; task < ntasks; task += PQ_THREADS / 32) {
      const int j = task / nparts, part = task - j * nparts;
      const int k0 = (int)((int64_t)part * K / nparts), k1 = (int)((int64_t)(part + 1) * K / nparts);
      const float4* xr = reinterpret_cast<const float4*>(sx + lane * pitch + j * dsub);
      const float4* cj = reinterpret_cast<const float4*>(cb + (int64_t)j * K * dsub);
      float best = -CUDART_INF_F;
      int besti = k0;
      for (int k = k0; k < k1; k += 2) {
        const bool two = k + 1 < k1;
        const float4* ca = cj + (int64_t)k * ds4;
        const float4* cbk = cj + (int64_t)(two ? k + 1 : k) * ds4;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f, b0 = 0.f, b1 = 0.f, b2 = 0.f, b3 = 0.f;
#pragma unroll 4
        for (int e = 0; e < ds4; ++e) {
          const float4 x = xr[e];
          const float4 u = __ldg(ca + e);
          const float4 v = __ldg(cbk + e);
          if (L2) {
            const float t0 = x.x - u.x, t1 = x.y - u.y, t2 = x.z - u.z, t3 = x.w - u.w;
            const float w0 = x.x - v.x, w1 = x.y - v.y, w2 = x.z - v.z, w3 = x.w - v.w;
            a0 = fmaf(t0, t0, a0); a1 = fmaf(t1, t1, a1); a2 = fmaf(t2, t2, a2); a3 = fmaf(t3, t3, a3);
            b0 = fmaf(w0, w0, b0); b1 = fmaf(w1, w1, b1); b2 = fmaf(w2, w2, b2); b3 = fmaf(w3, w3, b3);
          } else {
            a0 = fmaf(x.x, u.x, a0); a1 = fmaf(x.y, u.y, a1); a2 = fmaf(x.z, u.z, a2); a3 = fmaf(x.w, u.w, a3);
            b0 = fmaf(x.x, v.x, b0); b1 = fmaf(x.y, v.y, b1); b2 = fmaf(x.z, v.z, b2); b3 = fmaf(x.w, v.w, b3);
          }
        }
        const float sa = (a0 + a1) + (a2 + a3), sb = (b0 + b1) + (b2 + b3);
        const float s0 = L2 ? -sa : sa, s1 = L2 ? -sb : sb;
        if (s0 > best) {  // strict: the lowest index wins exact ties
          best = s0;
          besti = k;
        }
        if (two && s1 > best) {
          best = s1;
          besti = k + 1;
        }
      }
      s_bs[task * PQ_ROWS + lane] = best;
      s_bi[task * PQ_ROWS + lane] = besti;
    }
    __syncthreads();
    for (int i = tid; i < PQ_ROWS * M; i += PQ_THREADS) {  // consecutive threads -> consecutive code words
      const int r = i / M, j = i - r * M;
      float best = s_bs[(j * nparts) * PQ_ROWS + r];
      int besti = s_bi[(j * nparts) * PQ_ROWS + r];
      for (int part = 1; part < nparts; ++part) {  // slices ascend in k: strict > keeps the lowest index on ties
        const float sc = s_bs[(j * nparts + part) * PQ_ROWS + r];
        if (sc > best) {
          best = sc;
          besti = s_bi[(j * nparts + part) * PQ_ROWS + r];
        }
      }
      if (r < rows) codes[(work_rows ? (int64_t)work_rows[r0 + r] : r0 + r) * M + j] = besti;
    }
  }
}

// Arbiter of the (row, sub-vector) pairs the wide-codebook tensor kernel (pq_tensor.cuh) could not decide: one warp per
// pair, lane = centroids lane, lane+32, ...; per centroid exactly the arithmetic of pq_encode_kernel (four FMA chains over
// the elements e = 0, 4, 8, ... combined as (a0 + a1) + (a2 + a3); lowest index on ties), so a re-decided pair gets the
// code the sub-vector kernel would give it.
template <bool L2>
__global__ void __launch_bounds__(256) pq_fix_pairs_kernel(const float* __restrict__ X, int d, const float* __restrict__ cb, int M,
                                                           int K, int dsub, int32_t* __restrict__ codes,
                                                           const uint32_t* __restrict__ pairs,
                                                           const unsigned long long* __restrict__ n_pairs_dev,
                                                           unsigned long long cap) {
  const unsigned long long n_pairs = *n_pairs_dev < cap ? *n_pairs_dev : cap;
  const int lane = threadIdx.x & 31;
  const int ds4 = dsub >> 2;
  const unsigned long long warps = (unsigned long long)gridDim.x * (blockDim.x >> 5);
  for (unsigned long long i = (unsigned long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < n_pairs; i += warps) {
    const uint32_t pr = pairs[i];
    const int64_t row = pr / (uint32_t)M;
    const int j = (int)(pr - (uint32_t)row * (uint32_t)M);
    const float4* xr = reinterpret_cast<const float4*>(X + row * d + j * dsub);
    const float4* cj = reinterpret_cast<const float4*>(cb + (int64_t)j * K * dsub);
    float best = -CUDART_INF_F;
    int besti = 0x7fffffff;
    for (int k = lane; k < K; k += 32) {
      const float4* ca = cj + (int64_t)k * ds4;
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
      for (int e = 0; e < ds4; ++e) {
        const float4 x = __ldg(xr + e);
        const float4 u = __ldg(ca + e);
        if (L2) {
          const float t0 = x.x - u.x, t1 = x.y - u.y, t2 = x.z - u.z, t3 = x.w - u.w;
          a0 = fmaf(t0, t0, a0); a1 = fmaf(t1, t1, a1); a2 = fmaf(t2, t2, a2); a3 = fmaf(t3, t3, a3);
        } else {
          a0 = fmaf(x.x, u.x, a0); a1 = fmaf(x.y, u.y, a1); a2 = fmaf(x.z, u.z, a2); a3 = fmaf(x.w, u.w, a3);
        }
      }
      const float sa = (a0 + a1) + (a2 + a3);
      const float s0 = L2 ? -sa : sa;
      if (s0 > best) {  // ascending k per lane, strict: the lowest index wins exact ties; NaN / -inf scores never win
        best = s0;
        besti = k;
      }
    }
    // warp argmax, lowest index among equal scores (no candidate above -inf: code 0, as in the sub-vector kernel)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ob = __shfl_xor_sync(MEVI_FULL_MASK, best, o);
      const int oi = __shfl_xor_sync(MEVI_FULL_MASK, besti, o);
      if (ob > best || (ob == best && oi < besti)) { best = ob; besti = oi; }
    }
    if (lane == 0) codes[row * M + j] = besti == 0x7fffffff ? 0 : besti;
  }
}

}  // namespace

static int launch_pq_kernel(mevi_ctx* ctx, const float* X, int64_t n, int d, const float* codebook, int M, int K, int metric,
                            int32_t* codes, const int32_t* work_rows, const int64_t* n_work_dev, cudaStream_t st,
                            const int* run_if = nullptr) {
  const int dsub = d / M;
  const int nparts = M >= PQ_THREADS / 32 ? 1 : (PQ_THREADS / 32) / M;
  const size_t smem = (size_t)PQ_ROWS * (d + 4) * sizeof(float) + (size_t)M * nparts * PQ_ROWS * 8;
  MEVI_REQUIRE(ctx, smem <= 220 * 1024, "embedding width %d too large for the row tile", d);
  const int64_t n_tiles = (n + PQ_ROWS - 1) / PQ_ROWS;
  const int per_sm = smem <= 112 * 1024 ? 2 : 1;
  const int64_t max_grid = (int64_t)ctx->sm_count * per_sm;
  const int grid = (int)(n_tiles < max_grid ? n_tiles : max_grid);
  if (metric == MEVI_METRIC_L2) {
    MEVI_CUDA(ctx, cudaFuncSetAttribute(pq_encode_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    pq_encode_kernel<true><<<grid, PQ_THREADS, smem, st>>>(X, n, d, codebook, M, K, dsub, codes, work_rows, n_work_dev, run_if);
  } else {
    MEVI_CUDA(ctx, cudaFuncSetAttribute(pq_encode_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    pq_encode_kernel<false><<<grid, PQ_THREADS, smem, st>>>(X, n, d, codebook, M, K, dsub, codes, work_rows, n_work_dev, run_if);
  }
  MEVI_CUDA(ctx, cudaGetLastError());
  MEVI_COUNT_LAUNCH(ctx, 1);
  return MEVI_OK;
}

// rows the tensor prefilter flagged (work list on the device), re-decided by the sub-vector kernel; n = upper bound
int mevi_pq_fix_launch(mevi_ctx* ctx, const float* X, int64_t n, int d, const float* pq_codebook, int M, int K, int metric,
                       int32_t* codes, const int32_t* work_rows, const int64_t* n_work_dev, cudaStream_t st) {
  // a launch sized for a few flagged rows per thousand; the kernel's tile loop covers whatever the list holds
  const int64_t bound = n < (int64_t)ctx->sm_count * 2 * PQ_ROWS ? n : (int64_t)ctx->sm_count * 2 * PQ_ROWS;
  return launch_pq_kernel(ctx, X, bound, d, pq_codebook, M, K, metric, codes, work_rows, n_work_dev, st);
}

// pairs (row * M + sub-vector) of the wide-codebook tensor kernel, re-decided in the sub-vector kernel's arithmetic; if the
// pair list overflowed (*overflow != 0) the whole matrix is redone by the sub-vector kernel instead
int mevi_pq_fix_pairs_launch(mevi_ctx* ctx, const float* X, int64_t n, int d, const float* pq_codebook, int M, int K, int metric,
                             int32_t* codes, const uint32_t* pairs, const unsigned long long* n_pairs_dev, unsigned long long cap,
                             const int* overflow, cudaStream_t st) {
  const int dsub = d / M;
  if (metric == MEVI_METRIC_L2)
    pq_fix_pairs_kernel<true><<<ctx->sm_count * 8, 256, 0, st>>>(X, d, pq_codebook, M, K, dsub, codes, pairs, n_pairs_dev, cap);
  else
    pq_fix_pairs_kernel<false><<<ctx->sm_count * 8, 256, 0, st>>>(X, d, pq_codebook, M, K, dsub, codes, pairs, n_pairs_dev, cap);
  MEVI_CUDA(ctx, cudaGetLastError());
  MEVI_COUNT_LAUNCH(ctx, 1);
  return launch_pq_kernel(ctx, X, n, d, pq_codebook, M, K, metric, codes, nullptr, nullptr, st, overflow);
}

namespace {
// padded[j][k][:] = 0 except columns [j*dsub, (j+1)*dsub) = codebook[j][k][:]: sub-vector centroids zero-padded to the
// full width have orthogonal supports across levels, so the RQ residual corrections vanish and the RQ kernel's argmin
// per level IS the PQ argmin per sub-vector
__global__ void pq_pad_codebook_kernel(const float* __restrict__ cb, int M, int K, int dsub, float* __restrict__ padded) {
  const int d = M * dsub;
  const int64_t total = (int64_t)M * K * d;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % d);
    const int64_t jk = i / d;
    const int j = (int)(jk / K);
    const int e = c - j * dsub;
    padded[i] = (e >= 0 && e < dsub) ? cb[jk * dsub + e] : 0.f;
  }
}
}  // namespace

extern "C" int mevi_pq_encode(mevi_ctx* ctx, const float* X, int64_t n, int d, const float* codebook, int M, int K,
                              int metric, int32_t* codes, void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  if (n <= 0) return MEVI_OK;
  MEVI_REQUIRE(ctx, X && codebook && codes, "NULL argument");
  MEVI_REQUIRE(ctx, metric == MEVI_METRIC_L2 || metric == MEVI_METRIC_IP, "bad metric %d", metric);
  MEVI_REQUIRE(ctx, d > 0 && M > 0 && K > 0 && d % M == 0, "embedding width %d is not a multiple of subvector_num %d", d, M);
  const int dsub = d / M;
  MEVI_REQUIRE(ctx, dsub % 4 == 0, "sub-vector width %d must be a multiple of 4", dsub);
  MEVI_REQUIRE(ctx, (reinterpret_cast<uintptr_t>(X) & 15) == 0 && (reinterpret_cast<uintptr_t>(codebook) & 15) == 0,
               "X and codebook must be 16-byte aligned");
  // Tensor route (M*K <= 128, the shapes the RQ kernel takes): K1 on the block-padded codebook - one HBM pass at
  // ~70 % of the roofline instead of an FP32-issue-bound pass at 6 % - with the sub-vector kernel below as the arbiter
  // of the rows its prefilter flags.  MEVI_PQ_TENSOR=0 keeps everything on the sub-vector kernel.
  const char* env = getenv("MEVI_PQ_TENSOR");
  if (!(env && atoi(env) == 0) && n >= 4096 && mevi_rq_tensor_supported(ctx, d, M, K, metric)) {
    float* padded = (float*)mevi_ws(ctx, WS_PQ_PAD, (size_t)M * K * d * sizeof(float));
    if (!padded) return MEVI_ERR_NOMEM;
    pq_pad_codebook_kernel<<<ctx->sm_count, 256, 0, st>>>(codebook, M, K, dsub, padded);
    MEVI_CUDA(ctx, cudaGetLastError());
    MEVI_COUNT_LAUNCH(ctx, 1);
    return mevi_rq_tensor_assign(ctx, X, n, d, padded, M, K, metric, codes, M, nullptr, nullptr, nullptr, codebook, nullptr, st);
  }
  // wide codebooks (K = 256, sub-vector width 32): the split-fp16 tensor kernel of pq_tensor.cuh
  if (!(env && atoi(env) == 0) && n >= 4096 && mevi_pq_tensor_supported(ctx, n, d, M, K, metric))
    return mevi_pq_tensor_encode(ctx, X, n, d, codebook, M, K, metric, codes, st);
  return launch_pq_kernel(ctx, X, n, d, codebook, M, K, metric, codes, nullptr, nullptr, st);
}
