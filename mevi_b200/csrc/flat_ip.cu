// flat_ip.cu — K2 exact flat inner-product search with fused threshold top-k.
//
// Replaces MEVI/faiss_search.py:13-21 with param='Flat' (faiss IndexFlatIP
// add + search: Q[nq,d].D[N,d]^T, k best per query, descending).
//
// This file holds the fp32 CUDA-core path (MODE_EXACT, small inputs, and the
// fallback of the tcgen05 prefilter in flat_tensor.cu).  Structure shared by
// both: documents are visited in chunks whose size grows geometrically.  A tile kernel scores a [128 queries x 128 docs] block and
// appends (score,id) to the query's candidate buffer only when the score is not
// below the query's running k-th best (tau, fixed during a chunk).  After each
// chunk a per-query compaction kernel sorts the buffer, keeps the k best and
// raises tau.  With randomly ordered documents a chunk that doubles the number
// of documents seen adds ~k candidates per query, so the append path is cold
// and the kernel is bound by the dense contraction (2*nq*N*d FLOP).  Buffers
// that would overflow (adversarially sorted input) set a flag and the search is
// re-run with chunks that always fit.
#include <math_constants.h>

#include "common.cuh"

namespace {

constexpr int FT_BM = 128, FT_BN = 128, FT_BK = 16, FT_THREADS = 256;

struct FlatState {
  float* tau;         // [nq]
  int* count;         // [nq]
  float* cand_score;  // [nq][capg]
  int32_t* cand_id;   // [nq][capg]  row index inside the shard
  int* overflow;      // [1]
  int capg;
};

// scores tile: queries [q0, q0+128) x docs [n0, n0+128), fp32 FMA, sequential over d
__global__ void __launch_bounds__(FT_THREADS) flat_tile_kernel(const float* __restrict__ Q, int nq,
                                                               const float* __restrict__ D, int64_t n_begin,
                                                               int64_t n_end, int d, FlatState stt) {
  __shared__ float sA[FT_BK][FT_BM + 4];
  __shared__ float sB[FT_BK][FT_BN + 4];
  __shared__ float s_tau[FT_BM];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;  // 16 x 16 threads, 8x8 outputs each
  const int q0 = blockIdx.y * FT_BM;
  const int64_t n0 = n_begin + (int64_t)blockIdx.x * FT_BN;
  if (tid < FT_BM) s_tau[tid] = (q0 + tid < nq) ? stt.tau[q0 + tid] : CUDART_INF_F;

  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  // each thread loads one float4 of A and one of B per k-chunk: row = tid/4 (+64), k4 = (tid%4)*4
  const int lrow = tid >> 2, lk = (tid & 3) * 4;
  for (int k0 = 0; k0 < d; k0 += FT_BK) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int r = lrow + 64 * h;
      float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
      if (q0 + r < nq && k0 + lk < d) a = ldg_f4(Q + (int64_t)(q0 + r) * d + k0 + lk);
      if (n0 + r < n_end && k0 + lk < d) b = ld_stream_f4(D + (n0 + r) * d + k0 + lk);
      sA[lk + 0][r] = a.x; sA[lk + 1][r] = a.y; sA[lk + 2][r] = a.z; sA[lk + 3][r] = a.w;
      sB[lk + 0][r] = b.x; sB[lk + 1][r] = b.y; sB[lk + 2][r] = b.z; sB[lk + 3][r] = b.w;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < FT_BK; ++kk) {
      float a[8], b[8];
      *reinterpret_cast<float4*>(&a[0]) = *reinterpret_cast<const float4*>(&sA[kk][ty * 8]);
      *reinterpret_cast<float4*>(&a[4]) = *reinterpret_cast<const float4*>(&sA[kk][ty * 8 + 4]);
      *reinterpret_cast<float4*>(&b[0]) = *reinterpret_cast<const float4*>(&sB[kk][tx * 8]);
      *reinterpret_cast<float4*>(&b[4]) = *reinterpret_cast<const float4*>(&sB[kk][tx * 8 + 4]);
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int q = q0 + ty * 8 + i;
    if (q >= nq) continue;
    const float tau = s_tau[ty * 8 + i];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int64_t row = n0 + tx * 8 + j;
      if (row < n_end && !(acc[i][j] < tau)) {
        const int slot = atomicAdd(&stt.count[q], 1);
        if (slot < stt.capg) {
          stt.cand_score[(int64_t)q * stt.capg + slot] = acc[i][j];
          stt.cand_id[(int64_t)q * stt.capg + slot] = (int32_t)row;
        } else {
          *stt.overflow = 1;
        }
      }
    }
  }
}

// one CTA per query: sort the candidate buffer, keep k, raise tau
__global__ void __launch_bounds__(256) flat_compact_kernel(FlatState stt, int k, int cap_sort) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* s_score = reinterpret_cast<float*>(smem_raw);
  int32_t* s_id = reinterpret_cast<int32_t*>(s_score + cap_sort);
  const int q = blockIdx.x;
  int cnt = stt.count[q];
  if (cnt > stt.capg) cnt = stt.capg;
  if (cnt <= k && cnt == 0) return;
  for (int i = threadIdx.x; i < cap_sort; i += blockDim.x) {
    if (i < cnt) {
      s_score[i] = stt.cand_score[(int64_t)q * stt.capg + i];
      s_id[i] = stt.cand_id[(int64_t)q * stt.capg + i];
    } else {
      s_score[i] = -CUDART_INF_F;
      s_id[i] = 0x7fffffff;
    }
  }
  __syncthreads();
  block_bitonic_sort<int32_t>(s_score, s_id, cap_sort);
  const int kept = cnt < k ? cnt : k;
  for (int i = threadIdx.x; i < kept; i += blockDim.x) {
    stt.cand_score[(int64_t)q * stt.capg + i] = s_score[i];
    stt.cand_id[(int64_t)q * stt.capg + i] = s_id[i];
  }
  if (threadIdx.x == 0) {
    stt.count[q] = kept;
    stt.tau[q] = (kept >= k) ? s_score[k - 1] : -CUDART_INF_F;
  }
}

__global__ void flat_init_kernel(FlatState stt, int nq) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nq) {
    stt.tau[i] = -CUDART_INF_F;
    stt.count[i] = 0;
  }
  if (i == 0) *stt.overflow = 0;
}

__global__ void flat_emit_kernel(FlatState stt, int nq, int k, int64_t id_base, float* __restrict__ scores,
                                 int64_t* __restrict__ ids) {
  const int q = blockIdx.x;
  const int cnt = stt.count[q] < k ? stt.count[q] : k;
  for (int i = threadIdx.x; i < k; i += blockDim.x) {
    if (i < cnt) {
      scores[(int64_t)q * k + i] = stt.cand_score[(int64_t)q * stt.capg + i];
      ids[(int64_t)q * k + i] = id_base + (int64_t)stt.cand_id[(int64_t)q * stt.capg + i];
    } else {
      scores[(int64_t)q * k + i] = -CUDART_INF_F;
      ids[(int64_t)q * k + i] = -1;
    }
  }
}

int pow2_at_least(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

}  // namespace

extern "C" int mevi_flat_ip_topk(mevi_ctx* ctx, const float* Q, int nq, const float* D, int64_t n, int d, int k,
                                 int64_t id_base, int mode, float* scores, int64_t* ids, void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  MEVI_REQUIRE(ctx, Q && scores && ids && (D || n == 0), "NULL argument");
  MEVI_REQUIRE(ctx, d > 0 && d % 4 == 0, "flat search needs d %% 4 == 0 (got %d)", d);
  MEVI_REQUIRE(ctx, k >= 1 && k <= 2048, "k must be in [1, 2048] (got %d)", k);
  MEVI_REQUIRE(ctx, n >= 0 && n < (int64_t)2147483647, "shard too large for int32 row ids");
  if (nq <= 0) return MEVI_OK;
  bool use_tensor = false;
  if (mode == MEVI_MODE_TENSOR) {
    if (!mevi_flat_tensor_supported(ctx, d, k))
      return mevi_set_error(ctx, MEVI_ERR_UNSUPPORTED, "tensor flat search unsupported for d=%d k=%d", d, k);
    use_tensor = true;
  } else if (mode == MEVI_MODE_AUTO) {
    use_tensor = mevi_flat_tensor_supported(ctx, d, k) && n >= 8192;
  }

  if (use_tensor) {
    int fell_back = 1;
    int rc = mevi_flat_tensor_search(ctx, Q, nq, D, n, d, k, id_base, scores, ids, &fell_back, st);
    if (rc != MEVI_OK) return rc;
    if (!fell_back) return MEVI_OK;
    // margin window overflowed or fp16 range exceeded: the fp32 path below computes the answer instead
  }

  const int capg = pow2_at_least(k) < 2048 ? 4096 : 8192;  // >= 2k, power of two for the sorter
  const size_t off_tau = 0;
  const size_t off_cnt = off_tau + (size_t)nq * sizeof(float);
  const size_t off_ovf = off_cnt + (size_t)nq * sizeof(int);
  const size_t off_cs = (off_ovf + sizeof(int) + 255) & ~size_t(255);
  const size_t off_ci = off_cs + (size_t)nq * capg * sizeof(float);
  const size_t total = off_ci + (size_t)nq * capg * sizeof(int32_t);
  char* ws = (char*)mevi_ws(ctx, WS_TOPK_AUX, total);
  if (!ws) return MEVI_ERR_NOMEM;
  FlatState stt;
  stt.tau = (float*)(ws + off_tau);
  stt.count = (int*)(ws + off_cnt);
  stt.overflow = (int*)(ws + off_ovf);
  stt.cand_score = (float*)(ws + off_cs);
  stt.cand_id = (int32_t*)(ws + off_ci);
  stt.capg = capg;
  const size_t smem_compact = (size_t)capg * 8;
  MEVI_CUDA(ctx, cudaFuncSetAttribute(flat_compact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_compact));

  for (int attempt = 0; attempt < 2; ++attempt) {
    const bool safe = attempt == 1;
    flat_init_kernel<<<(nq + 255) / 256, 256, 0, st>>>(stt, nq);
    MEVI_COUNT_LAUNCH(ctx, 1);
    MEVI_CUDA(ctx, cudaGetLastError());
    const int64_t first = ((capg - k) / FT_BN) * FT_BN;  // a chunk this small can never overflow
    int64_t chunk = first;
    int64_t pos = 0;
    while (pos < n) {
      int64_t end = pos + chunk < n ? pos + chunk : n;
      {
        dim3 grid((unsigned)((end - pos + FT_BN - 1) / FT_BN), (unsigned)((nq + FT_BM - 1) / FT_BM));
        flat_tile_kernel<<<grid, FT_THREADS, 0, st>>>(Q, nq, D, pos, end, d, stt);
        MEVI_COUNT_LAUNCH(ctx, 1);
        MEVI_CUDA(ctx, cudaGetLastError());
      }
      flat_compact_kernel<<<nq, 256, smem_compact, st>>>(stt, k, capg);
      MEVI_COUNT_LAUNCH(ctx, 1);
      MEVI_CUDA(ctx, cudaGetLastError());
      pos = end;
      if (!safe) {
        // documents seen so far = pos; a chunk of 3x that adds ~3k expected candidates per query
        int64_t next = pos * 3;
        const int64_t cap_chunk = (int64_t)1 << 22;
        chunk = next < first ? first : (next > cap_chunk ? cap_chunk : next);
        chunk = (chunk / FT_BN) * FT_BN;
      }
    }
    int h_overflow = 0;
    MEVI_CUDA(ctx, cudaMemcpyAsync(&h_overflow, stt.overflow, sizeof(int), cudaMemcpyDeviceToHost, st));
    MEVI_CUDA(ctx, cudaStreamSynchronize(st));
    if (!h_overflow) break;
    if (safe) return mevi_set_error(ctx, MEVI_ERR_CUDA, "flat search candidate buffer overflowed in safe mode");
  }
  flat_emit_kernel<<<nq, 128, 0, st>>>(stt, nq, k, id_base, scores, ids);
  MEVI_COUNT_LAUNCH(ctx, 1);
  MEVI_CUDA(ctx, cudaGetLastError());
  return MEVI_OK;
}
