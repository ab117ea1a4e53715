// rq_tensor.cu — K1: tcgen05/TMEM residual-quantisation encode + k-means assignment.
//
// Replaces the arithmetic of MEVI/pq.py:281-305 (and the assignment half of 551-598) for the
// shipped shape family (d % 64 == 0, K % 32 == 0, M*K <= 128).
//
// Algebraic form.  The reference subtracts the chosen centroid after every level, so level j sees
// r_j = x - sum_{m<j} c^m_{k_m}.  Distances to level-j centroids only need
//     r_j . c^j_k = x . c^j_k - sum_{m<j} (c^m_{k_m} . c^j_k)
// so ONE contraction X[rows,d] . C_all[M*K,d]^T serves all levels; the second term comes from a
// precomputed cross-level Gram table.  X is read from HBM exactly once (4*d bytes per row).
//
// Precision.  The tensor result is only a PREFILTER with a rigorous error bound; whatever it cannot decide is
// re-decided with more precision, and rows that stay inside the tightest bound go to a work list for the fp32
// direct-form kernel of rq_exact.cu, the literal restatement of the reference arithmetic.  Rows outside the bounds
// provably have the same argmin in exact arithmetic, so codes agree with the reference except at fp32-epsilon ties.
// The kernel (rq_tensor4.cuh, generation 4) contracts in split fp16, hi.hi + hi.lo + lo.hi (22 significant bits,
// ~2^-22 |x||c| error), with the document operand in tensor memory; it runs the M = 1 k-means assignment at the HBM
// roofline and the M = 4 encode at 0.62-0.69 of it (tensor work under the power cap).  DESIGN.md section 4 has the
// measurements that led here, including those of the slower alternatives.
// Roofline: HBM (4*d B/row).
#include <cuda.h>
#include <cuda_fp16.h>
#include <math_constants.h>

#include "common.cuh"
#include "ptx.cuh"

namespace {

constexpr int CONV_WARP0 = 4, CONV_WARPS = 8, EPI_WARP0 = 12;
constexpr int TMEM_COLS = 512;
constexpr float U_REL = 1.0f / 524288.0f;    // 2^-19: relative bound on the contraction error (|x||c| units)

enum { C_SC = 0, C_SX, C_INV, C_INV_SX2, C_FX, C_FC, C_NUM = 8 };

struct Params {
  const float* X; int64_t n; int d; int nchunks;
  int M, K, NT, N1, metric;
  const __half* Bimg; const float* cn2; const float* e1; const float* lvl; const float* gram; const float* consts;
  int gram_floats;
  int32_t* codes; int64_t codes_stride;
  int32_t* work_rows; int32_t* work_levels; unsigned long long* work_count;
  // fused k-means pass (rq_tensor4_kernel<1, true>): previous assignment in, per-CTA partial sums | counts out
  const int32_t* prev; int64_t prev_stride; float* part_sums; int32_t* part_counts;
  double* inertia; int* err_flag;
  int64_t n_tiles;
};

// ---- preparation kernels ---------------------------------------------------------------------
__global__ void absmax_kernel(const float* __restrict__ p, int64_t rows, int d, int64_t row_step, unsigned* out) {
  // max |v| over rows 0, row_step, 2*row_step, ...   (non-negative floats order like their bit patterns)
  unsigned m = 0;
  const int64_t nsel = (rows + row_step - 1) / row_step;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nsel * d; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = (i / d) * row_step;
    const float v = fabsf(p[r * d + (i % d)]);
    if (v == v && v < CUDART_INF_F) m = max(m, __float_as_uint(v));
  }
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(MEVI_FULL_MASK, m, o));
  if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}

__device__ __forceinline__ float pow2_scale(float amax) {
  // 2^s with amax * 2^s in [2^13, 2^14): two bits of headroom below the fp16 maximum
  if (!(amax > 0.f)) return 1.f;
  return ldexpf(1.f, 13 - ilogbf(amax));
}

__global__ void consts_kernel(const unsigned* absmax2, int d, float* consts) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    const float sc = pow2_scale(__uint_as_float(absmax2[0]));
    const float sx = pow2_scale(__uint_as_float(absmax2[1]));
    consts[C_SC] = sc;
    consts[C_SX] = sx;
    consts[C_INV] = 1.f / (sc * sx);
    consts[C_INV_SX2] = (1.f / sx) * (1.f / sx);
    const float floor_abs = sqrtf((float)d) * 5.9604645e-8f;  // sqrt(d) * 2^-24: fp16 subnormal spacing of hi+lo
    consts[C_FX] = floor_abs / sx;
    consts[C_FC] = floor_abs / sc;
  }
}

// one warp per centroid row: squared norm (double accumulation)
__global__ void cnorm_kernel(const float* __restrict__ cb, int rows_valid, int d, int NT, float* __restrict__ cn2,
                             float* __restrict__ cnorm) {
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= NT) return;
  double s = 0.0;
  if (r < rows_valid)
    for (int c = threadIdx.x & 31; c < d; c += 32) {
      const double v = cb[(size_t)r * d + c];
      s += v * v;
    }
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(MEVI_FULL_MASK, s, o);
  if ((threadIdx.x & 31) == 0) {
    cn2[r] = (float)s;
    cnorm[r] = (float)sqrt(s);
  }
}

// gram[(level j block) + prow*K + k] = c_prow . c^j_k   for prow in [0, j*K); one warp per entry
__global__ void gram_kernel(const float* __restrict__ cb, int M, int K, int d, float* __restrict__ gram, int total) {
  const int e = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (e >= total) return;
  int j = 1, off = 0;
  while (e >= off + j * K * K) {
    off += j * K * K;
    ++j;
  }
  const int loc = e - off;
  const int prow = loc / K, k = loc - prow * K;
  const float* a = cb + (size_t)prow * d;
  const float* b = cb + ((size_t)j * K + k) * d;
  double s = 0.0;
  for (int c = threadIdx.x & 31; c < d; c += 32) s += (double)a[c] * (double)b[c];
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(MEVI_FULL_MASK, s, o);
  if ((threadIdx.x & 31) == 0) gram[e] = (float)s;
}


// Error model of the prefilter (all in distance units; f = 2 for L2 where dist = |c|^2 - 2 dot, 1 for IP):
//   |dist_k - exact| <= |x| * E1_k + B_j/2,
//   E1_k = f (U_REL + EPS_A) |c_k| + f Fc      contraction error + fp16 floor of the codebook + fp32 epilogue
//   B_j  = 2 [ f Fx cmax_j + EPS_A (c2max_j + f j gmax_j) ]   fp16 floor of x + roundings of |c|^2 and Gram terms
// A (row, level) is decided by the prefilter only if  d_other - |x| E1_other > d_best + |x| E1_best + B_j
// for every other candidate; otherwise the exact kernel re-decides it.  One block per level.
__global__ void level_consts_kernel(const float* __restrict__ cnorm, const float* __restrict__ cn2,
                                    const float* __restrict__ gram, int M, int K, int metric,
                                    const float* __restrict__ consts, float* __restrict__ e1, float* __restrict__ lvl) {
  const int j = blockIdx.x, lane = threadIdx.x;
  const float f = metric == MEVI_METRIC_L2 ? 2.f : 1.f;
  const float EPS_A = 4.8e-7f;  // 2^-21
  float cmax = 0.f, c2max = 0.f, gmax = 0.f;
  for (int k = lane; k < K; k += 32) {
    const float cn = cnorm[j * K + k];
    cmax = fmaxf(cmax, cn);
    c2max = fmaxf(c2max, cn2[j * K + k]);
    e1[j * K + k] = f * (U_REL + EPS_A) * cn + f * consts[C_FC];
  }
  if (j > 0) {
    const float* gj = gram + (size_t)(j * (j - 1) / 2) * K * K;
    for (int i = lane; i < j * K * K; i += 32) gmax = fmaxf(gmax, fabsf(gj[i]));
  }
  for (int o = 16; o > 0; o >>= 1) {
    cmax = fmaxf(cmax, __shfl_xor_sync(MEVI_FULL_MASK, cmax, o));
    c2max = fmaxf(c2max, __shfl_xor_sync(MEVI_FULL_MASK, c2max, o));
    gmax = fmaxf(gmax, __shfl_xor_sync(MEVI_FULL_MASK, gmax, o));
  }
  if (lane == 0) {
    lvl[j * 4 + 0] = 0.f;
    lvl[j * 4 + 1] = 2.f * (f * consts[C_FX] * cmax + EPS_A * (c2max + f * (float)j * gmax));
    lvl[j * 4 + 2] = cmax;
    lvl[j * 4 + 3] = gmax;
  }
}

__global__ void finish_stats_kernel(const unsigned long long* work_count, int64_t rows, int64_t* stats) {
  if (threadIdx.x == 0 && blockIdx.x == 0 && stats) {
    atomicAdd((unsigned long long*)&stats[0], *work_count);
    atomicAdd((unsigned long long*)&stats[1], (unsigned long long)rows);
  }
}

// residual[row] = ((x - c0) - c1) - ...   in the reference's order (pq.py:304-305)
__global__ void residual_from_codes_kernel(const float* __restrict__ X, int64_t n, int d4, const float* __restrict__ cb,
                                           int M, int K, const int32_t* __restrict__ codes, int64_t codes_stride,
                                           float* __restrict__ residual) {
  const int64_t total = n * d4;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / d4;
    const int c = (int)(i - row * d4);
    float4 v = reinterpret_cast<const float4*>(X)[i];
    for (int m = 0; m < M; ++m) {
      const int code = codes[row * codes_stride + m];
      const float4 cc = __ldg(reinterpret_cast<const float4*>(cb) + ((int64_t)m * K + code) * d4 + c);
      v.x -= cc.x; v.y -= cc.y; v.z -= cc.z; v.w -= cc.w;
    }
    reinterpret_cast<float4*>(residual)[i] = v;
  }
}

// Bimg32[chunk][row][32 halfs] per 32-wide K chunk, rows 0..NT-1 = hi(c*sc), NT..2NT-1 = lo; 16-byte units XOR-swizzled
// by (row>>1)&3 (the UMMA 64-byte swizzle).  The hi rows of a chunk are one contiguous NT*64-byte block.
constexpr int KC32 = 32;
__global__ void bimg32_kernel(const float* __restrict__ cb, int rows_valid, int d, int NT, const float* __restrict__ consts,
                              __half* __restrict__ Bimg) {
  const int units_per_row = d / 8;
  const int total = NT * units_per_row;
  const float sc = consts[C_SC];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int r = i / units_per_row, ug = i - r * units_per_row;
    const int chunk = ug / 4, u = ug & 3;
    __half hi[8], lo[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float t = r < rows_valid ? cb[(size_t)r * d + ug * 8 + e] * sc : 0.f;
      hi[e] = __float2half_rn(t);
      lo[e] = __float2half_rn(t - __half2float(hi[e]));
    }
    const size_t base = (size_t)chunk * (2 * NT) * KC32;
    const int up = u ^ ((r >> 1) & 3);  // NT % 8 == 0, so row NT + r has the same swizzle phase
    *reinterpret_cast<uint4*>(Bimg + base + (size_t)r * KC32 + up * 8) = *reinterpret_cast<const uint4*>(hi);
    *reinterpret_cast<uint4*>(Bimg + base + (size_t)(NT + r) * KC32 + up * 8) = *reinterpret_cast<const uint4*>(lo);
  }
}

// after the encode kernel: a pipeline time-out (err != 0) must never leave plausible-looking codes behind
__global__ void poison_codes_kernel(const int* __restrict__ err, int32_t* __restrict__ codes, int64_t n, int64_t stride, int M) {
  if (*err == 0) return;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n * M; i += (int64_t)gridDim.x * blockDim.x)
    codes[(i / M) * stride + (i % M)] = -1;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// 2-D tensor map over X[n][d] fp32 with a [box_rows x 32 floats] box, 128B-swizzled (one box row = one 128-byte line)
inline int make_x_tensormap(mevi_ctx* ctx, const float* X, int64_t n, int d, int box_rows, CUtensorMap* out,
                            CUtensorMapL2promotion promo = CU_TENSOR_MAP_L2_PROMOTION_L2_256B, int box_cols = KC32) {
  if (!ctx->tmap_encode_fn) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn ||
        qres != cudaDriverEntryPointSuccess) {
      cudaGetLastError();
      return mevi_set_error(ctx, MEVI_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
    }
    ctx->tmap_encode_fn = fn;
  }
  const cuuint64_t gdim[2] = {(cuuint64_t)d, (cuuint64_t)n};
  const cuuint64_t gstride[1] = {(cuuint64_t)d * 4};
  const cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};  // rows narrower than 128 B: no swizzle
  const cuuint32_t estr[2] = {1, 1};
  CUresult r = ((EncodeTiledFn)ctx->tmap_encode_fn)(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)X, gdim, gstride, box, estr,
                                                    CU_TENSOR_MAP_INTERLEAVE_NONE,
                                                    box_cols == KC32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE, promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return mevi_set_error(ctx, MEVI_ERR_CUDA, "cuTensorMapEncodeTiled (128B swizzle, %d-row box) failed with %d", box_rows, (int)r);
  return MEVI_OK;
}

#include "rq_tensor4.cuh"
#include "pq_tensor.cuh"

bool shape_ok(mevi_ctx* ctx, int d, int M, int K, int metric) {
  if (!ctx || ctx->cc_major != 10) return false;
  if (d < 64 || d % 64 != 0 || d > 8192) return false;
  if (M < 1 || M > 4 || K < 32 || K % 32 != 0) return false;
  const int NT = M * K;
  if (NT > 128 || NT % 16 != 0) return false;
  return metric == MEVI_METRIC_L2 || metric == MEVI_METRIC_IP;
}

}  // namespace

// fused k-means pass: the [K][d] accumulators must fit next to a 3-stage fp32 ring
bool mevi_kmeans_fused_supported(mevi_ctx* ctx, int d, int K) {
  if (!shape_ok(ctx, d, 1, K, MEVI_METRIC_L2)) return false;
  if (K > 32 || K % v4::ACC_WARPS != 0 || d % KC32 != 0) return false;
  return v4::smem4_layout(1, K, K, K * d).total + 1024 <= 227 * 1024;
}

bool mevi_rq_tensor_supported(mevi_ctx* ctx, int d, int M, int K, int metric) {
  if (!shape_ok(ctx, d, M, K, metric)) return false;
  const int NT = M * K;
  return v4::smem4_layout(M, K, NT).total + 1024 <= 227 * 1024;
}

int mevi_rq_tensor_assign(mevi_ctx* ctx, const float* X, int64_t n, int d, const float* cb, int M, int K, int metric,
                          int32_t* codes, int64_t codes_stride, float* residual, int64_t* stats, double* inertia,
                          const float* pq_codebook, const KmeansFusedPass* km_fused, cudaStream_t st) {
  if (!mevi_rq_tensor_supported(ctx, d, M, K, metric))
    return mevi_set_error(ctx, MEVI_ERR_UNSUPPORTED, "tensor RQ path unsupported for d=%d M=%d K=%d", d, M, K);
  MEVI_REQUIRE(ctx, (reinterpret_cast<uintptr_t>(X) & 15) == 0 && (reinterpret_cast<uintptr_t>(cb) & 15) == 0,
               "X and codebook must be 16-byte aligned");
  if (n <= 0) return MEVI_OK;
  // a pipeline time-out in an earlier (asynchronous) launch is reported here at the latest; mevi_ctx_check reports it on demand
  if (int rc = mevi_deferred_error(ctx)) return rc;
  const int NT = M * K, N1 = 2 * NT, nchunks = d / KC32;
  int gram_floats = 0;
  for (int j = 1; j < M; ++j) gram_floats += j * K * K;
  // ---- scratch: [consts | absmax2 | work_count | cn2 | cnorm | e1 | lvl | gram | Bimg]
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = (off + bytes + 255) & ~size_t(255); return o; };
  const size_t o_consts = take(C_NUM * 4), o_abs = take(8), o_cnt = take(8), o_cn2 = take(NT * 4),
               o_cnorm = take(NT * 4), o_e1 = take(NT * 4), o_lvl = take(8 * 4 * 4),
               o_gram = take((size_t)(gram_floats ? gram_floats : 1) * 4),
               o_bimg = take((size_t)nchunks * N1 * KC32 * 2 + 1024);
  char* ws = (char*)mevi_ws(ctx, WS_RQ_PREP, off);
  if (!ws) return MEVI_ERR_NOMEM;
  float* consts = (float*)(ws + o_consts);
  unsigned* absmax2 = (unsigned*)(ws + o_abs);
  unsigned long long* work_count = (unsigned long long*)(ws + o_cnt);
  float* cn2 = (float*)(ws + o_cn2);
  float* cnorm = (float*)(ws + o_cnorm);
  float* lvl = (float*)(ws + o_lvl);
  float* e1 = (float*)(ws + o_e1);
  float* gram = (float*)(ws + o_gram);
  __half* Bimg = (__half*)(ws + o_bimg);
  int32_t* work = (int32_t*)mevi_ws(ctx, WS_RQ_WORK, (size_t)n * 8);
  if (!work) return MEVI_ERR_NOMEM;
  int* err_flag = ctx->dev_err + MEVI_ERRSLOT_RQ;

  MEVI_CUDA(ctx, cudaMemsetAsync(ws + o_abs, 0, o_cn2 - o_abs, st));  // absmax2, work count
  absmax_kernel<<<32, 256, 0, st>>>(cb, (int64_t)M * K, d, 1, absmax2);
  const int64_t sample_rows = 2048;
  const int64_t row_step = n > sample_rows ? n / sample_rows : 1;
  absmax_kernel<<<ctx->sm_count, 256, 0, st>>>(X, n, d, row_step, absmax2 + 1);
  consts_kernel<<<1, 32, 0, st>>>(absmax2, d, consts);
  bimg32_kernel<<<(NT * (d / 8) + 255) / 256, 256, 0, st>>>(cb, M * K, d, NT, consts, Bimg);
  cnorm_kernel<<<(NT + 7) / 8, 256, 0, st>>>(cb, M * K, d, NT, cn2, cnorm);
  if (gram_floats) gram_kernel<<<(gram_floats + 7) / 8, 256, 0, st>>>(cb, M, K, d, gram, gram_floats);
  level_consts_kernel<<<M, 32, 0, st>>>(cnorm, cn2, gram, M, K, metric, consts, e1, lvl);
  MEVI_CUDA(ctx, cudaGetLastError());
  MEVI_COUNT_LAUNCH(ctx, gram_floats ? 7 : 6);

  Params p;
  p.X = X; p.n = n; p.d = d; p.nchunks = nchunks; p.M = M; p.K = K; p.NT = NT; p.N1 = N1; p.metric = metric;
  p.Bimg = Bimg; p.cn2 = cn2; p.e1 = e1; p.lvl = lvl; p.gram = gram; p.consts = consts; p.gram_floats = gram_floats;
  p.codes = codes; p.codes_stride = codes_stride;
  p.work_rows = work; p.work_levels = work + n; p.work_count = work_count;
  p.inertia = inertia; p.err_flag = err_flag;
  p.prev = nullptr; p.prev_stride = 0; p.part_sums = nullptr; p.part_counts = nullptr;
  CUtensorMap tmap;
  int trc = make_x_tensormap(ctx, X, n, d, v4::TM4, &tmap);
  if (trc != MEVI_OK) return trc;
  p.n_tiles = (n + v4::TM4 - 1) / v4::TM4;
  const size_t smem4 = (size_t)v4::smem4_layout(M, K, NT).total + 1024;
  const int grid4 = (int)(p.n_tiles < ctx->sm_count ? p.n_tiles : ctx->sm_count);
#define MEVI_LAUNCH_RQ_TENSOR4(MM)                                                                                          \
  do {                                                                                                                      \
    MEVI_CUDA(ctx, cudaFuncSetAttribute(v4::rq_tensor4_kernel<MM, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem4)); \
    v4::rq_tensor4_kernel<MM, false><<<grid4, v4::THREADS4, smem4, st>>>(p, tmap);                                          \
  } while (0)
  if (km_fused != nullptr && M == 1) {
    // fused k-means pass: assignment + accumulation under the previous assignment in one read of the shard
    if (!mevi_kmeans_fused_supported(ctx, d, K))
      return mevi_set_error(ctx, MEVI_ERR_UNSUPPORTED, "fused k-means pass unsupported for d=%d K=%d", d, K);
    p.prev = km_fused->prev; p.prev_stride = km_fused->prev_stride;
    p.part_sums = km_fused->part_sums; p.part_counts = km_fused->part_counts;
    const size_t smem_acc = (size_t)v4::smem4_layout(1, K, NT, K * d).total + 1024;
    MEVI_CUDA(ctx, cudaFuncSetAttribute(v4::rq_tensor4_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_acc));
    v4::rq_tensor4_kernel<1, true><<<grid4, v4::THREADS4_ACC, smem_acc, st>>>(p, tmap);
  } else
  switch (M) {
    case 1: MEVI_LAUNCH_RQ_TENSOR4(1); break;
    case 2: MEVI_LAUNCH_RQ_TENSOR4(2); break;
    case 3: MEVI_LAUNCH_RQ_TENSOR4(3); break;
    default: MEVI_LAUNCH_RQ_TENSOR4(4); break;
  }
#undef MEVI_LAUNCH_RQ_TENSOR4
  MEVI_CUDA(ctx, cudaGetLastError());
  poison_codes_kernel<<<ctx->sm_count, 256, 0, st>>>(err_flag, codes, n, codes_stride, M);
  MEVI_COUNT_LAUNCH(ctx, 2);
  if (int rc = mevi_publish_errors(ctx, st)) return rc;

  // exact re-decision of the flagged rows (count stays on the device): the fp32 direct-form RQ kernel, or - when this
  // is a PQ encode running on a block-padded codebook - the sub-vector kernel, so that flagged rows get exactly the
  // codes mevi_pq_encode's CUDA-core path gives them
  int rc;
  if (pq_codebook != nullptr && codes_stride == M)
    rc = mevi_pq_fix_launch(ctx, X, n, d, pq_codebook, M, K, metric, codes, work,
                            reinterpret_cast<const int64_t*>(work_count), st);
  else
    rc = mevi_rq_exact_launch(ctx, X, n, d, cb, M, K, metric, codes, codes_stride, nullptr, work, work + n,
                              reinterpret_cast<const int64_t*>(work_count), n, nullptr, st);
  if (rc != MEVI_OK) return rc;
  if (stats) {
    finish_stats_kernel<<<1, 32, 0, st>>>(work_count, n, stats);
    MEVI_COUNT_LAUNCH(ctx, 1);
  }
  if (residual) {
    residual_from_codes_kernel<<<ctx->sm_count * 16, 256, 0, st>>>(X, n, d / 4, cb, M, K, codes, codes_stride, residual);
    MEVI_COUNT_LAUNCH(ctx, 1);
  }
  MEVI_CUDA(ctx, cudaGetLastError());
  return MEVI_OK;
}

// ---- wide-codebook PQ encode (pq_tensor.cuh) ---------------------------------------------------------------------
bool mevi_pq_tensor_supported(mevi_ctx* ctx, int64_t n, int d, int M, int K, int metric) {
  if (!ctx || ctx->cc_major != 10) return false;
  if (K != pq256::KQ || M < 1 || (d != M * 32 && d != M * 24)) return false;
  if (n * (int64_t)M >= (int64_t)1 << 32) return false;  // pair ids are 32-bit
  return metric == MEVI_METRIC_L2 || metric == MEVI_METRIC_IP;
}

int mevi_pq_tensor_encode(mevi_ctx* ctx, const float* X, int64_t n, int d, const float* cb, int M, int K, int metric,
                          int32_t* codes, cudaStream_t st) {
  if (!mevi_pq_tensor_supported(ctx, n, d, M, K, metric))
    return mevi_set_error(ctx, MEVI_ERR_UNSUPPORTED, "tensor PQ path unsupported for d=%d M=%d K=%d", d, M, K);
  if (n <= 0) return MEVI_OK;
  if (int rc = mevi_deferred_error(ctx)) return rc;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = (off + bytes + 255) & ~size_t(255); return o; };
  const size_t o_consts = take(C_NUM * 4), o_abs = take(8), o_cnt = take(8), o_ovf = take(8), o_subc = take((size_t)M * 16 + 64),
               o_bimg = take((size_t)M * pq256::B_SUBQ);
  char* ws = (char*)mevi_ws(ctx, WS_RQ_PREP, off);
  if (!ws) return MEVI_ERR_NOMEM;
  const unsigned long long cap = (unsigned long long)(n * (int64_t)M / 8 + 65536);
  uint32_t* pairs = (uint32_t*)mevi_ws(ctx, WS_RQ_WORK, (size_t)cap * 4);
  if (!pairs) return MEVI_ERR_NOMEM;
  float* consts = (float*)(ws + o_consts);
  unsigned* absmax2 = (unsigned*)(ws + o_abs);
  unsigned long long* pair_count = (unsigned long long*)(ws + o_cnt);
  int* overflow = (int*)(ws + o_ovf);
  float* subc = (float*)(ws + o_subc);
  __half* Bimg = (__half*)(ws + o_bimg);
  int* err_flag = ctx->dev_err + MEVI_ERRSLOT_RQ;

  MEVI_CUDA(ctx, cudaMemsetAsync(ws + o_abs, 0, o_subc - o_abs, st));  // absmax2, pair count, overflow flag
  const int ds = d / M;
  absmax_kernel<<<32, 256, 0, st>>>(cb, (int64_t)M * K, ds, 1, absmax2);
  const int64_t sample_rows = 2048;
  const int64_t row_step = n > sample_rows ? n / sample_rows : 1;
  absmax_kernel<<<ctx->sm_count, 256, 0, st>>>(X, n, d, row_step, absmax2 + 1);
  pq256::pq_scale_kernel<<<1, 32, 0, st>>>(absmax2, ds, consts);
  pq256::pq_bimg_kernel<<<(M * K * 4 + 255) / 256, 256, 0, st>>>(cb, M, ds, metric, consts, Bimg);
  pq256::pq_consts_kernel<<<M, pq256::KQ, 0, st>>>(cb, ds, metric, consts, subc);
  MEVI_CUDA(ctx, cudaGetLastError());

  pq256::PqParams p;
  p.X = X; p.n = n; p.d = d; p.M = M; p.metric = metric;
  p.Bimg = Bimg; p.subc = subc; p.consts = consts;
  p.codes = codes; p.pairs = pairs; p.pair_count = pair_count; p.pair_cap = cap; p.overflow = overflow;
  p.err_flag = err_flag;
  p.n_tiles = (n + pq256::TMQ - 1) / pq256::TMQ;
  CUtensorMap tmap;
  // 128-byte L2 promotion: a pass reads 384-byte row pieces, 256-byte promotion would fetch 512
  int trc = make_x_tensormap(ctx, X, n, d, pq256::TMQ, &tmap, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, ds);
  if (trc != MEVI_OK) return trc;
  const size_t smem = (size_t)pq256::smemq_layout().total + 1024;
  const int grid = (int)(p.n_tiles < ctx->sm_count ? p.n_tiles : ctx->sm_count);
  if (ds == 32) {
    MEVI_CUDA(ctx, cudaFuncSetAttribute(pq256::pq_tensor_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    pq256::pq_tensor_kernel<32><<<grid, pq256::THREADSQ, smem, st>>>(p, tmap);
  } else {
    MEVI_CUDA(ctx, cudaFuncSetAttribute(pq256::pq_tensor_kernel<24>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    pq256::pq_tensor_kernel<24><<<grid, pq256::THREADSQ, smem, st>>>(p, tmap);
  }
  MEVI_CUDA(ctx, cudaGetLastError());
  poison_codes_kernel<<<ctx->sm_count, 256, 0, st>>>(err_flag, codes, n, M, M);
  MEVI_COUNT_LAUNCH(ctx, 7);
  if (int rc = mevi_publish_errors(ctx, st)) return rc;
  return mevi_pq_fix_pairs_launch(ctx, X, n, d, cb, M, K, metric, codes, pairs, pair_count, cap, overflow, st);
}
