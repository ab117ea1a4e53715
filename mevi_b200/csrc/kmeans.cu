// kmeans.cu — full-batch Lloyd pieces: per-centroid sum/count accumulation,
// centroid update, residual update.
//
// Reference behaviour being replaced: MEVI/pq.py:551-598 trains each RQ level
// with sklearn MiniBatchKMeans on rank 0 and subtracts centers[pred] in numpy
// (591-593).  BASELINE.json asks for the data-parallel form instead: every rank
// assigns its row block, accumulates [K,d] sums and [K] counts, and one
// all-reduce(SUM) of the fused [K*d+K] buffer (precedent: pq.py:384-397)
// gives every rank the same new centroids.
//
// Accumulation is DETERMINISTIC: a CTA walks a contiguous range of rows in
// tiles; inside a tile rows are bucketed by centroid with a stable counting
// sort, and every (centroid, column) accumulator is a register owned by one
// thread that adds the bucket's rows in ascending row order.  Per-CTA partials
// are then reduced in a fixed order.  No float atomics, so sums are
// bit-reproducible for a given (n, grid) and ranks stay in lockstep.
// Roofline: HBM (one more read of the shard: 4*d bytes per row + 4 B assignment).

#include <cub/cub.cuh>

#include "common.cuh"
#include "ptx.cuh"

namespace {

constexpr int KM_THREADS = 256;
constexpr int KM_WARPS = KM_THREADS / 32;
constexpr int KM_TILE = 256;
constexpr int KA_MAX_STAGES = 8;
constexpr int KA_DEFAULT_STAGES = 2;  // shared-memory stages of the accumulate kernel (stages-1 bulk copies in flight)
static_assert(KA_DEFAULT_STAGES >= 2 && KA_DEFAULT_STAGES <= KA_MAX_STAGES, "the accumulate kernel's barrier arrays hold KA_MAX_STAGES");

// Column-owner accumulation (skew-proof and deterministic).  The CTA keeps the running [K][d] fp32
// sums in shared memory; thread t owns column t of every centroid.  Rows arrive in sub-tiles — one
// contiguous byte range, fetched with a single bulk async copy (TMA engine) into a double-buffered
// shared-memory stage.  Every thread then walks the sub-tile's rows in order and adds its column to
// the accumulator row of the row's centroid (a CTA-uniform index, so the access stays conflict-free).
// All threads work on every row, so one dominant cluster (the reference-trained codebooks put >80 %
// of N(0,1) rows into two centroids) costs nothing extra; the summation order is the row order.
template <int NT>  // NT column-owner threads + one loader warp
__global__ void __launch_bounds__(NT + 32, 1) kmeans_accumulate_kernel(const float* __restrict__ R, int64_t n, int d,
                                                                       const int32_t* __restrict__ assign,
                                                                       int64_t assign_stride, int K, int sub_rows,
                                                                       int KA_STAGES,
                                                                       float* __restrict__ partial_sums,     // [grid][K][d]
                                                                       int32_t* __restrict__ partial_counts)  // [grid][K]
{
  extern __shared__ __align__(128) unsigned char km_smem[];  // [KA_STAGES][sub_rows][d] fp32, then acc [K][d]
  __shared__ __align__(8) uint64_t full_bar[KA_MAX_STAGES];
  __shared__ __align__(8) uint64_t empty_bar[KA_MAX_STAGES];
  __shared__ int s_assign[KA_MAX_STAGES][32];
  __shared__ int s_count_total[64];

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool owner = tid < d;  // this thread owns column tid of every centroid's running sum
  // sub-tiles are dealt round-robin (CTA b takes sub-tiles b, b+G, ...): neighbouring SMs stream
  // neighbouring memory, like the encode kernel; the per-CTA order is still fixed -> reproducible
  const int64_t total_sub = (n + sub_rows - 1) / sub_rows;
  const int64_t nsub = total_sub > blockIdx.x ? (total_sub - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  const int64_t row_end = n;
  const size_t stage_bytes = (size_t)sub_rows * d * sizeof(float);
  float* s_acc = reinterpret_cast<float*>(km_smem + KA_STAGES * stage_bytes);

  for (int i = tid; i < K * d; i += NT + 32) s_acc[i] = 0.f;
  for (int i = tid; i < 64; i += NT + 32) s_count_total[i] = 0;
  if (tid == 0) {
    for (int s = 0; s < KA_STAGES; ++s) {
      ptx::mbar_init(&full_bar[s], 1);
      ptx::mbar_init(&empty_bar[s], NT / 32);
    }
    ptx::mbar_fence_init();
  }
  __syncthreads();
  // No CTA-wide barrier inside the loop: the loader warp runs ahead (assignment loads from global memory and the bulk
  // copy of the rows are both off the owners' critical path), owners drift freely and hand stages back per warp.
  if (warp == NT / 32) {
    for (int64_t i = 0; i < nsub; ++i) {
      const int s = (int)(i % KA_STAGES);
      const int64_t r0 = (blockIdx.x + i * gridDim.x) * sub_rows;
      const int rows = (int)((row_end - r0) < sub_rows ? (row_end - r0) : sub_rows);
      int a = 0;
      if (lane < rows) {  // issued before the wait: the load latency overlaps it
        a = assign[(r0 + lane) * assign_stride];
        a = a < 0 ? 0 : (a >= K ? K - 1 : a);
      }
      if (i >= KA_STAGES) ptx::mbar_wait_backoff(&empty_bar[s], (uint32_t)(((i / KA_STAGES) - 1) & 1), 32);
      if (lane < rows) {
        s_assign[s][lane] = a;
        atomicAdd(&s_count_total[a], 1);
      }
      __syncwarp();
      if (lane == 0) {
        const uint32_t bytes = (uint32_t)rows * (uint32_t)d * 4u;
        ptx::mbar_arrive_expect_tx(&full_bar[s], bytes);
        ptx::bulk_g2s(km_smem + (size_t)s * stage_bytes, R + r0 * d, bytes, &full_bar[s]);
      }
    }
  } else {
    float* my_acc = s_acc + tid;
    for (int64_t i = 0; i < nsub; ++i) {
      const int64_t r0 = (blockIdx.x + i * gridDim.x) * sub_rows;
      const int rows = (int)((row_end - r0) < sub_rows ? (row_end - r0) : sub_rows);
      const int stg = (int)(i % KA_STAGES);
      ptx::mbar_wait(&full_bar[stg], (uint32_t)((i / KA_STAGES) & 1));
      if (owner) {
        const float* base = reinterpret_cast<const float*>(km_smem + (size_t)stg * stage_bytes) + tid;
        const int* as = s_assign[stg];
        // the row's centroid is a CTA-uniform value, so the dynamically indexed accumulator row costs
        // nothing in shared memory; rows are added in order -> the sum is reproducible
        for (int r = 0; r < rows; ++r) my_acc[(size_t)as[r] * d] += base[(size_t)r * d];
      }
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&empty_bar[stg]);
    }
  }
  __syncthreads();
  for (int i = tid; i < K * d; i += NT + 32) partial_sums[(int64_t)blockIdx.x * K * d + i] = s_acc[i];
  if (tid < K) partial_counts[(int64_t)blockIdx.x * K + tid] = s_count_total[tid];
}

// generic fallback (any K, d % 4 == 0): warp per row, float atomics into sums
__global__ void kmeans_accumulate_atomic_kernel(const float* __restrict__ R, int64_t n, int d,
                                                const int32_t* __restrict__ assign, int64_t assign_stride, int K,
                                                float* __restrict__ sums, float* __restrict__ counts) {
  const int lane = threadIdx.x & 31;
  const int64_t warp_global = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t row = warp_global; row < n; row += n_warps) {
    int a = assign[row * assign_stride];
    a = a < 0 ? 0 : (a >= K ? K - 1 : a);
    for (int c = lane; c < d; c += 32) atomicAdd(&sums[(int64_t)a * d + c], R[row * d + c]);
    if (lane == 0) atomicAdd(&counts[a], 1.0f);
  }
}

__global__ void kmeans_reduce_partials_kernel(const float* __restrict__ partial_sums,
                                              const int32_t* __restrict__ partial_counts, int G, int K, int d,
                                              float* __restrict__ sums_counts) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t kd = (int64_t)K * d;
  if (i < kd) {
    float s = 0.f;
    for (int g = 0; g < G; ++g) s += partial_sums[(int64_t)g * kd + i];  // fixed order
    sums_counts[i] = s;
  } else if (i < kd + K) {
    const int k = (int)(i - kd);
    long long c = 0;
    for (int g = 0; g < G; ++g) c += partial_counts[(int64_t)g * K + k];
    sums_counts[i] = (float)c;
  }
}

__global__ void kmeans_update_kernel(const float* __restrict__ sums_counts, int K, int d, float* __restrict__ centroids,
                                     int32_t* __restrict__ n_empty) {
  const int64_t kd = (int64_t)K * d;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < kd) {
    const int k = (int)(i / d);
    const float cnt = sums_counts[kd + k];
    if (cnt > 0.f) centroids[i] = sums_counts[i] / cnt;
  }
  if (n_empty && i < K) {
    if (!(sums_counts[kd + i] > 0.f)) atomicAdd(n_empty, 1);
  }
}

__global__ void residual_update_kernel(float* __restrict__ R, int64_t n, int d4, const float* __restrict__ centroids,
                                       int K, const int32_t* __restrict__ assign, int64_t assign_stride) {
  const int64_t total = n * d4;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / d4;
    const int c = (int)(i - row * d4);
    int a = assign[row * assign_stride];
    a = a < 0 ? 0 : (a >= K ? K - 1 : a);
    float4 v = reinterpret_cast<float4*>(R)[i];
    const float4 cc = __ldg(reinterpret_cast<const float4*>(centroids) + (int64_t)a * d4 + c);
    v.x -= cc.x; v.y -= cc.y; v.z -= cc.z; v.w -= cc.w;
    reinterpret_cast<float4*>(R)[i] = v;
  }
}

template <int NT>
cudaError_t launch_accumulate_nt(const float* R, int64_t n, int d, const int32_t* assign, int64_t stride, int K, int G,
                                 float* ps, int32_t* pc, int sub_rows, int stages, size_t smem, cudaStream_t st) {
  cudaError_t e = cudaFuncSetAttribute(kmeans_accumulate_kernel<NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  kmeans_accumulate_kernel<NT><<<G, NT + 32, smem, st>>>(R, n, d, assign, stride, K, sub_rows, stages, ps, pc);
  return cudaGetLastError();
}

cudaError_t launch_accumulate(const float* R, int64_t n, int d, const int32_t* assign, int64_t stride, int K, int G,
                              float* ps, int32_t* pc, int sub_rows, int stages, size_t smem, cudaStream_t st) {
  // one thread per column
  if (d <= 128) return launch_accumulate_nt<128>(R, n, d, assign, stride, K, G, ps, pc, sub_rows, stages, smem, st);
  if (d <= 256) return launch_accumulate_nt<256>(R, n, d, assign, stride, K, G, ps, pc, sub_rows, stages, smem, st);
  if (d <= 512) return launch_accumulate_nt<512>(R, n, d, assign, stride, K, G, ps, pc, sub_rows, stages, smem, st);
  if (d <= 768) return launch_accumulate_nt<768>(R, n, d, assign, stride, K, G, ps, pc, sub_rows, stages, smem, st);
  return launch_accumulate_nt<992>(R, n, d, assign, stride, K, G, ps, pc, sub_rows, stages, smem, st);
}

// per-centroid sums|counts of the rows of R under a given assignment -> sums_counts [K*d + K]
int accumulate_by_code(mevi_ctx* ctx, const float* R, int64_t n, int d, const int32_t* assign, int64_t stride, int K,
                       float* sums_counts, cudaStream_t st) {
  const int64_t kd = (int64_t)K * d;
  // shared-memory budget: [K][d] accumulators + KA_STAGES stages of sub_rows rows
  const size_t acc_bytes = (size_t)kd * sizeof(float);
  const int KA_STAGES = KA_DEFAULT_STAGES;
  int sub_rows = acc_bytes + 4096 < 220 * 1024 ? (int)((220 * 1024 - acc_bytes) / ((size_t)KA_STAGES * d * 4)) : 0;
  if (sub_rows > 32) sub_rows = 32;
  const bool fast = K <= 64 && d <= 992 && d % 4 == 0 && sub_rows >= 4 && (reinterpret_cast<uintptr_t>(R) & 15) == 0;
  if (fast) {
    int G = ctx->sm_count;  // one CTA per SM (shared-memory stages), persistent
    int64_t max_g = (n + sub_rows - 1) / sub_rows;
    if (G > max_g) G = (int)max_g;
    if (G < 1) G = 1;
    size_t ps_bytes = (size_t)G * kd * sizeof(float);
    size_t pc_bytes = (size_t)G * K * sizeof(int32_t);
    char* ws = (char*)mevi_ws(ctx, WS_KM_PARTIAL, ps_bytes + pc_bytes);
    if (!ws) return MEVI_ERR_NOMEM;
    float* ps = (float*)ws;
    int32_t* pc = (int32_t*)(ws + ps_bytes);
    const size_t smem = (size_t)KA_STAGES * sub_rows * d * 4 + acc_bytes + 128;
    cudaError_t e = launch_accumulate(R, n, d, assign, stride, K, G, ps, pc, sub_rows, KA_STAGES, smem, st);
    if (e != cudaSuccess) return mevi_set_error(ctx, MEVI_ERR_CUDA, "kmeans_accumulate launch: %s", cudaGetErrorString(e));
    int threads = 256;
    int blocks = (int)((kd + K + threads - 1) / threads);
    kmeans_reduce_partials_kernel<<<blocks, threads, 0, st>>>(ps, pc, G, K, d, sums_counts);
    MEVI_COUNT_LAUNCH(ctx, 2);
    MEVI_CUDA(ctx, cudaGetLastError());
  } else {
    MEVI_CUDA(ctx, cudaMemsetAsync(sums_counts, 0, (size_t)(kd + K) * sizeof(float), st));
    int grid = ctx->sm_count * 8;
    kmeans_accumulate_atomic_kernel<<<grid, 256, 0, st>>>(R, n, d, assign, stride, K, sums_counts, sums_counts + kd);
    MEVI_COUNT_LAUNCH(ctx, 1);
    MEVI_CUDA(ctx, cudaGetLastError());
  }
  return MEVI_OK;
}


// ---- incremental Lloyd iteration: move only the rows whose assignment changed -------------------------------------
// sums_t[k] = sums_{t-1}[k] + (rows that moved to k) - (rows that moved away from k).  The running sums | counts live in
// float64 ("master"), so repeated corrections do not drift; the corrections themselves are fresh fp32 sums per CTA over
// a contiguous slice of the (ascending) list of changed rows, thread = column, rows in list order - no float atomics,
// bit-reproducible.  Per-CTA partials are folded into the master in CTA order.
struct ChangedPred {
  const int32_t* prev; int64_t pstride; const int32_t* cur; int64_t cstride;
  __host__ __device__ __forceinline__ bool operator()(const int& i) const {
    return prev[(int64_t)i * pstride] != cur[(int64_t)i * cstride];
  }
};

// (row, old centroid | new centroid << 16) per changed row: one 8-byte record, so the accumulation kernel's loads
// depend on ONE earlier load instead of three
__global__ void kmeans_delta_pack_kernel(const int32_t* __restrict__ prev, int64_t pstride, const int32_t* __restrict__ cur,
                                         int64_t cstride, const int32_t* __restrict__ changed, const int* __restrict__ n_changed,
                                         int K, int2* __restrict__ packed) {
  const int64_t m = *n_changed;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = changed[i];
    const int ko = min(max(prev[row * pstride], 0), K - 1), kn = min(max(cur[row * cstride], 0), K - 1);
    packed[i] = make_int2((int)row, ko | (kn << 16));
  }
}

// thread = column; a CTA walks a contiguous slice of the packed list in chunks of DELTA_CHUNK records staged in shared
// memory; rows go through a two-stage register pipeline (8 rows being added while the next 8 are in flight), and the
// register budget leaves room for two CTAs per SM
constexpr int DELTA_CHUNK = 256, DELTA_U = 8;

__global__ void __launch_bounds__(1024, 2)
kmeans_delta_kernel(const float* __restrict__ R, int d, const int2* __restrict__ packed, const int* __restrict__ n_changed,
                    int K, float* __restrict__ part_sums, int32_t* __restrict__ part_counts) {
  extern __shared__ float s_acc[];  // [K][d] signed sums of this CTA's slice
  __shared__ int s_cnt[256];        // [K] signed counts (K <= 256)
  __shared__ int2 s_rec[DELTA_CHUNK];
  const int col = threadIdx.x;      // blockDim.x >= d, one column per thread
  const bool live = col < d;
  const int64_t m = *n_changed;
  const int64_t lo = m * blockIdx.x / gridDim.x, hi = m * (blockIdx.x + 1) / gridDim.x;
  if (live)
    for (int k = 0; k < K; ++k) s_acc[k * d + col] = 0.f;
  for (int k = threadIdx.x; k < K; k += blockDim.x) s_cnt[k] = 0;  // (a narrow slice has fewer threads than centroids)
  const float* Rc = R + (live ? col : 0);

  auto fetch = [&](float (&v)[DELTA_U], int b0, int nrec) {
#pragma unroll
    for (int j = 0; j < DELTA_U; ++j) v[j] = (b0 + j < nrec && live) ? __ldg(Rc + (int64_t)s_rec[b0 + j].x * d) : 0.f;
  };
  auto add = [&](const float (&v)[DELTA_U], int b0, int nrec) {
#pragma unroll
    for (int j = 0; j < DELTA_U; ++j) {
      if (b0 + j >= nrec) break;
      const int kk = s_rec[b0 + j].y;
      const int ko = kk & 0xFFFF, kn = kk >> 16;
      if (live) {
        s_acc[kn * d + col] += v[j];
        s_acc[ko * d + col] -= v[j];
      }
      if (threadIdx.x == 0) { s_cnt[kn] += 1; s_cnt[ko] -= 1; }
    }
  };

  for (int64_t c0 = lo; c0 < hi; c0 += DELTA_CHUNK) {
    const int nrec = (int)((hi - c0) < DELTA_CHUNK ? (hi - c0) : DELTA_CHUNK);
    __syncthreads();  // the previous chunk's records are no longer read (and the zeroing above is complete)
    for (int t = threadIdx.x; t < nrec; t += blockDim.x) s_rec[t] = __ldg(&packed[c0 + t]);
    __syncthreads();
    float va[DELTA_U], vb[DELTA_U];
    fetch(va, 0, nrec);
    for (int b0 = 0; b0 < nrec; b0 += 2 * DELTA_U) {
      fetch(vb, b0 + DELTA_U, nrec);
      add(va, b0, nrec);
      fetch(va, b0 + 2 * DELTA_U, nrec);
      add(vb, b0 + DELTA_U, nrec);
    }
  }
  __syncthreads();
  if (live)
    for (int k = 0; k < K; ++k) part_sums[((int64_t)blockIdx.x * K + k) * d + col] = s_acc[k * d + col];
  for (int k = threadIdx.x; k < K; k += blockDim.x) part_counts[(int64_t)blockIdx.x * K + k] = s_cnt[k];
}

// master (float64) += the partials in CTA order; sums_counts = (float) master
__global__ void kmeans_delta_fold_kernel(const float* __restrict__ part_sums, const int32_t* __restrict__ part_counts, int G,
                                         int K, int d, double* __restrict__ master, float* __restrict__ sums_counts) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t kd = (int64_t)K * d;
  if (i < kd) {
    double a = master[i];
    for (int g = 0; g < G; ++g) a += (double)part_sums[(int64_t)g * kd + i];
    master[i] = a;
    sums_counts[i] = (float)a;
  } else if (i < kd + K) {
    const int k = (int)(i - kd);
    long long c = 0;
    for (int g = 0; g < G; ++g) c += part_counts[(int64_t)g * K + k];
    const double a = master[i] + (double)c;
    master[i] = a;
    sums_counts[i] = (float)a;
  }
}

}  // namespace

extern "C" {

int mevi_kmeans_step(mevi_ctx* ctx, const float* R, int64_t n, int d, const float* centroids, int K, int mode,
                     int32_t* assign_out_or_null, int64_t assign_stride, float* sums_counts, double* inertia_or_null,
                     void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  MEVI_REQUIRE(ctx, R && centroids && sums_counts, "NULL argument");
  MEVI_REQUIRE(ctx, n >= 0 && d > 0 && d % 4 == 0 && d <= 1024 && K >= 1, "unsupported shape n=%lld d=%d K=%d",
               (long long)n, d, K);
  MEVI_REQUIRE(ctx, n < (int64_t)2147483647, "shard too large for int32 row ids");
  int32_t* assign = assign_out_or_null;
  int64_t stride = assign_stride;
  if (!assign) {
    assign = (int32_t*)mevi_ws(ctx, WS_KM_ASSIGN, (size_t)(n > 0 ? n : 1) * sizeof(int32_t));
    if (!assign) return MEVI_ERR_NOMEM;
    stride = 1;
  }
  MEVI_REQUIRE(ctx, stride >= 1, "assign_stride must be >= 1");
  if (inertia_or_null) MEVI_CUDA(ctx, cudaMemsetAsync(inertia_or_null, 0, sizeof(double), st));
  const int64_t kd = (int64_t)K * d;
  if (n == 0) {
    MEVI_CUDA(ctx, cudaMemsetAsync(sums_counts, 0, (size_t)(kd + K) * sizeof(float), st));
    return MEVI_OK;
  }
  // 1. assignment
  bool use_tensor = false;
  if (mode == MEVI_MODE_TENSOR) {
    if (!mevi_rq_tensor_supported(ctx, d, 1, K, MEVI_METRIC_L2))
      return mevi_set_error(ctx, MEVI_ERR_UNSUPPORTED, "tensor k-means assignment unsupported for d=%d K=%d", d, K);
    use_tensor = true;
  } else if (mode == MEVI_MODE_AUTO) {
    use_tensor = mevi_rq_tensor_supported(ctx, d, 1, K, MEVI_METRIC_L2) && n >= 4096;
  }
  int rc;
  if (use_tensor)
    rc = mevi_rq_tensor_assign(ctx, R, n, d, centroids, 1, K, MEVI_METRIC_L2, assign, stride, nullptr, nullptr,
                               inertia_or_null, nullptr, nullptr, st);
  else
    rc = mevi_rq_exact_launch(ctx, R, n, d, centroids, 1, K, MEVI_METRIC_L2, assign, stride, nullptr, nullptr, nullptr,
                              nullptr, n, inertia_or_null, st);
  if (rc != MEVI_OK) return rc;

  // 2. accumulation
  rc = accumulate_by_code(ctx, R, n, d, assign, stride, K, sums_counts, st);
  if (rc != MEVI_OK) return rc;
  return MEVI_OK;
}

int mevi_kmeans_step_fused(mevi_ctx* ctx, const float* R, int64_t n, int d, const float* centroids, int K,
                           const int32_t* prev_assign, int64_t prev_stride, int32_t* assign_out, int64_t assign_stride,
                           float* sums_counts_prev, double* inertia_or_null, void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  MEVI_REQUIRE(ctx, R && centroids && prev_assign && assign_out && sums_counts_prev, "NULL argument");
  MEVI_REQUIRE(ctx, prev_stride >= 1 && assign_stride >= 1, "strides must be >= 1");
  MEVI_REQUIRE(ctx, n > 0 && n < (int64_t)2147483647, "n out of range");
  if (!mevi_kmeans_fused_supported(ctx, d, K) || n < 4096)
    return mevi_set_error(ctx, MEVI_ERR_UNSUPPORTED, "fused k-means pass unsupported for n=%lld d=%d K=%d (use mevi_kmeans_step)",
                          (long long)n, d, K);
  if (inertia_or_null) MEVI_CUDA(ctx, cudaMemsetAsync(inertia_or_null, 0, sizeof(double), st));
  const int64_t kd = (int64_t)K * d;
  const int64_t n_tiles = (n + 255) / 256;
  const int G = (int)(n_tiles < ctx->sm_count ? n_tiles : ctx->sm_count);  // the kernel's grid: one partial per CTA
  const size_t ps_bytes = (size_t)G * kd * sizeof(float), pc_bytes = (size_t)G * K * sizeof(int32_t);
  char* ws = (char*)mevi_ws(ctx, WS_KM_PARTIAL, ps_bytes + pc_bytes);
  if (!ws) return MEVI_ERR_NOMEM;
  const KmeansFusedPass fused = {prev_assign, prev_stride, (float*)ws, (int32_t*)(ws + ps_bytes)};
  const int rc = mevi_rq_tensor_assign(ctx, R, n, d, centroids, 1, K, MEVI_METRIC_L2, assign_out, assign_stride, nullptr, nullptr,
                                       inertia_or_null, nullptr, &fused, st);
  if (rc != MEVI_OK) return rc;
  const int threads = 256;
  kmeans_reduce_partials_kernel<<<(int)((kd + K + threads - 1) / threads), threads, 0, st>>>((const float*)ws, (const int32_t*)(ws + ps_bytes),
                                                                                             G, K, d, sums_counts_prev);
  MEVI_COUNT_LAUNCH(ctx, 1);
  MEVI_CUDA(ctx, cudaGetLastError());
  return MEVI_OK;
}


int mevi_kmeans_step_delta(mevi_ctx* ctx, const float* R, int64_t n, int d, const float* centroids, int K, int mode,
                           const int32_t* prev_assign, int64_t prev_stride, int32_t* assign_out, int64_t assign_stride,
                           double* master_sums_counts, float* sums_counts, int32_t* n_changed_or_null,
                           double* inertia_or_null, void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  MEVI_REQUIRE(ctx, R && centroids && prev_assign && assign_out && master_sums_counts && sums_counts, "NULL argument");
  MEVI_REQUIRE(ctx, prev_assign != assign_out, "prev_assign and assign_out must be different buffers");
  MEVI_REQUIRE(ctx, prev_stride >= 1 && assign_stride >= 1, "strides must be >= 1");
  MEVI_REQUIRE(ctx, n > 0 && n < (int64_t)2147483647 && d > 0 && d % 4 == 0 && d <= 1024 && K >= 1,
               "unsupported shape n=%lld d=%d K=%d", (long long)n, d, K);
  const int64_t kd = (int64_t)K * d;
  const size_t smem = (size_t)kd * sizeof(float);
  if (K > 256 || smem > 200 * 1024)  // (codes are packed 16 + 16 bits)
    return mevi_set_error(ctx, MEVI_ERR_UNSUPPORTED, "incremental k-means step unsupported for K=%d d=%d (use mevi_kmeans_step)", K, d);
  if (inertia_or_null) MEVI_CUDA(ctx, cudaMemsetAsync(inertia_or_null, 0, sizeof(double), st));
  // 1. assignment under the current centroids (the one pass over the shard)
  bool use_tensor = false;
  if (mode == MEVI_MODE_TENSOR) {
    if (!mevi_rq_tensor_supported(ctx, d, 1, K, MEVI_METRIC_L2))
      return mevi_set_error(ctx, MEVI_ERR_UNSUPPORTED, "tensor k-means assignment unsupported for d=%d K=%d", d, K);
    use_tensor = true;
  } else if (mode == MEVI_MODE_AUTO) {
    use_tensor = mevi_rq_tensor_supported(ctx, d, 1, K, MEVI_METRIC_L2) && n >= 4096;
  }
  int rc;
  if (use_tensor)
    rc = mevi_rq_tensor_assign(ctx, R, n, d, centroids, 1, K, MEVI_METRIC_L2, assign_out, assign_stride, nullptr, nullptr,
                               inertia_or_null, nullptr, nullptr, st);
  else
    rc = mevi_rq_exact_launch(ctx, R, n, d, centroids, 1, K, MEVI_METRIC_L2, assign_out, assign_stride, nullptr, nullptr, nullptr,
                              nullptr, n, inertia_or_null, st);
  if (rc != MEVI_OK) return rc;
  // 2. ascending list of the rows whose assignment changed (count stays on the device)
  const int G = ctx->sm_count * 2;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = (off + bytes + 255) & ~size_t(255); return o; };
  const size_t o_cnt = take(16), o_list = take((size_t)n * sizeof(int32_t)), o_pack = take((size_t)n * sizeof(int2)),
               o_ps = take((size_t)G * kd * sizeof(float)), o_pc = take((size_t)G * K * sizeof(int32_t));
  char* ws = (char*)mevi_ws(ctx, WS_KM_PARTIAL, off);
  if (!ws) return MEVI_ERR_NOMEM;
  int* d_count = (int*)(ws + o_cnt);
  int32_t* list = (int32_t*)(ws + o_list);
  int2* packed = (int2*)(ws + o_pack);
  float* ps = (float*)(ws + o_ps);
  int32_t* pc = (int32_t*)(ws + o_pc);
  ChangedPred pred{prev_assign, prev_stride, assign_out, assign_stride};
  cub::CountingInputIterator<int> ids(0);
  size_t tmp_bytes = 0;
  MEVI_CUDA(ctx, cub::DeviceSelect::If(nullptr, tmp_bytes, ids, list, d_count, (int)n, pred, st));
  void* tmp = mevi_ws(ctx, WS_SORT_TMP, tmp_bytes);
  if (!tmp) return MEVI_ERR_NOMEM;
  MEVI_CUDA(ctx, cub::DeviceSelect::If(tmp, tmp_bytes, ids, list, d_count, (int)n, pred, st));
  // 3. signed sums of the changed rows, folded into the float64 master
  const int threads = ((d + 31) / 32) * 32;
  MEVI_CUDA(ctx, cudaFuncSetAttribute(kmeans_delta_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kmeans_delta_pack_kernel<<<ctx->sm_count * 4, 256, 0, st>>>(prev_assign, prev_stride, assign_out, assign_stride, list, d_count, K,
                                                               packed);
  kmeans_delta_kernel<<<G, threads, smem, st>>>(R, d, packed, d_count, K, ps, pc);
  kmeans_delta_fold_kernel<<<(int)((kd + K + 255) / 256), 256, 0, st>>>(ps, pc, G, K, d, master_sums_counts, sums_counts);
  if (n_changed_or_null)
    MEVI_CUDA(ctx, cudaMemcpyAsync(n_changed_or_null, d_count, sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
  MEVI_CUDA(ctx, cudaGetLastError());
  MEVI_COUNT_LAUNCH(ctx, 4);
  return MEVI_OK;
}

int mevi_accumulate_by_code(mevi_ctx* ctx, const float* X, int64_t n, int d, const int32_t* assign, int64_t assign_stride,
                            int K, float* sums_counts, void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  MEVI_REQUIRE(ctx, X && assign && sums_counts, "NULL argument");
  MEVI_REQUIRE(ctx, n >= 0 && d > 0 && d % 4 == 0 && d <= 1024 && K >= 1 && assign_stride >= 1,
               "unsupported shape n=%lld d=%d K=%d", (long long)n, d, K);
  if (n == 0) {
    MEVI_CUDA(ctx, cudaMemsetAsync(sums_counts, 0, (size_t)((int64_t)K * d + K) * sizeof(float), st));
    return MEVI_OK;
  }
  return accumulate_by_code(ctx, X, n, d, assign, assign_stride, K, sums_counts, st);
}

int mevi_kmeans_update(mevi_ctx* ctx, const float* sums_counts, int K, int d, float* centroids, int32_t* n_empty_or_null,
                       void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  MEVI_REQUIRE(ctx, sums_counts && centroids && K >= 1 && d >= 1, "bad argument");
  if (n_empty_or_null) MEVI_CUDA(ctx, cudaMemsetAsync(n_empty_or_null, 0, sizeof(int32_t), st));
  const int64_t kd = (int64_t)K * d;
  int threads = 256;
  int blocks = (int)((kd + threads - 1) / threads);
  kmeans_update_kernel<<<blocks, threads, 0, st>>>(sums_counts, K, d, centroids, n_empty_or_null);
  MEVI_COUNT_LAUNCH(ctx, 1);
  MEVI_CUDA(ctx, cudaGetLastError());
  return MEVI_OK;
}

int mevi_residual_update(mevi_ctx* ctx, float* R, int64_t n, int d, const float* centroids, int K, const int32_t* assign,
                         int64_t assign_stride, void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  MEVI_REQUIRE(ctx, R && centroids && assign && d > 0 && d % 4 == 0 && K >= 1 && assign_stride >= 1, "bad argument");
  if (n <= 0) return MEVI_OK;
  int grid = ctx->sm_count * 16;
  residual_update_kernel<<<grid, 256, 0, st>>>(R, n, d / 4, centroids, K, assign, assign_stride);
  MEVI_COUNT_LAUNCH(ctx, 1);
  MEVI_CUDA(ctx, cudaGetLastError());
  return MEVI_OK;
}

}  // extern "C"
