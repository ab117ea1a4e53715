// common.cuh — context, error plumbing and warp helpers shared by every kernel file.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>

#include "../../include/mevi_b200.h"

#define MEVI_WARP 32
#define MEVI_FULL_MASK 0xffffffffu

enum WsSlot {
  WS_RQ_PREP = 0,   // tensor path: packed fp16 codebook image, norms, gram
  WS_RQ_WORK,       // tensor path: flagged-row worklist
  WS_KM_PARTIAL,    // k-means: per-CTA partial sums
  WS_KM_ASSIGN,     // k-means: assignment scratch when the caller passes none
  WS_TOPK_PART,     // re-rank / flat: per-split partial top-k lists
  WS_TOPK_AUX,      // flat: thresholds, counters, candidate buffers
  WS_SORT_TMP,      // inverted lists: radix sort temp
  WS_SORT_KEYS,     // inverted lists: unsorted keys / ids
  WS_HOST_STAGE_A,  // device staging for the host-buffer encode (double buffered)
  WS_HOST_STAGE_B,
  WS_HOST_CODES_A,
  WS_HOST_CODES_B,
  WS_MISC,
  WS_PQ_PAD,        // PQ encode on the tensor path: block-padded codebook
  WS_FLAT_IMAGE,    // one-shot flat search: fp16 image of the documents (+ its metadata)
  WS_GR_PLAN,       // grouped re-rank: device-side round plan (counts, scans, arrival numbers)
  WS_GR_MC,         // grouped re-rank of a multi-cluster index: per-query leaf tables, prefilter factors, margins
  WS_RA_PLAN,       // grouped rerank_all: pairs by leaf, work-item scan
  WS_RA_SORT,       // candidate sort: keys, values (double buffered), chunk offsets
  WS_NUM
};

struct mevi_ctx {
  int device = 0;
  int sm_count = 0;
  int cc_major = 0, cc_minor = 0;
  size_t total_mem = 0;
  size_t l2_bytes = 0;
  std::string err;
  void* ws[WS_NUM] = {nullptr};
  size_t ws_bytes[WS_NUM] = {0};
  void* pinned[4] = {nullptr, nullptr, nullptr, nullptr};
  size_t pinned_bytes[4] = {0, 0, 0, 0};
  cudaStream_t aux_stream[2] = {nullptr, nullptr};
  cudaEvent_t aux_event[4] = {nullptr, nullptr, nullptr, nullptr};
  void* tmap_encode_fn = nullptr;  // cuTensorMapEncodeTiled, resolved lazily
  // Device-side error words (a bounded mbarrier wait that times out sets one and the kernel bails out) and their
  // pinned host mirror.  Asynchronous entry points copy dev_err -> host_err at the end of their launch sequence;
  // the mirror is inspected at the start of the next call, after every synchronising call, and by mevi_ctx_check.
  int* dev_err = nullptr;            // [MEVI_ERRSLOTS]
  volatile int* host_err = nullptr;  // [MEVI_ERRSLOTS], cudaMallocHost
  // host-side state of the grouped re-rank's round plan between mevi_rerank_grouped_plan and its _plan_fill calls
  // (rerank_plan.cu owns the layout; malloc'ed, freed with the context)
  void* gr_plan = nullptr;
  // host-side state of a multi-cluster grouped call between mevi_rerank_grouped_multiclus and its _finish (flat_tensor.cu)
  void* gr_mc = nullptr;
  int64_t launches = 0;            // kernels launched by this context (reported by mevi_device_info)
};

enum { MEVI_ERRSLOT_RQ = 0, MEVI_ERRSLOT_RERANK = 1, MEVI_ERRSLOT_OTHER = 2, MEVI_ERRSLOTS = 8 };

int mevi_set_error(mevi_ctx* ctx, int code, const char* fmt, ...);
// enqueue the dev_err -> host_err copy on `st` (end of an asynchronous launch sequence)
int mevi_publish_errors(mevi_ctx* ctx, cudaStream_t st);
// MEVI_OK, or MEVI_ERR_CUDA (message set, error words cleared) if a kernel of an earlier launch reported a time-out
int mevi_deferred_error(mevi_ctx* ctx);
// grow-on-demand scratch; returns nullptr (and sets the error) on failure
void* mevi_ws(mevi_ctx* ctx, int slot, size_t bytes);
void* mevi_pinned(mevi_ctx* ctx, int slot, size_t bytes);

// ---- internal entry points called across kernel files (the C ABI is include/mevi_b200.h) ----------------------
// rq_exact.cu: fp32 direct-form RQ encode / k-means assignment, of all rows or of the rows of a device-side work list
int mevi_rq_exact_launch(mevi_ctx* ctx, const float* X, int64_t n, int d, const float* cb, int M, int K, int metric,
                         int32_t* codes, int64_t codes_stride, float* residual, const int32_t* work_rows,
                         const int32_t* work_levels, const int64_t* n_work_dev, int64_t n_items, double* inertia,
                         cudaStream_t st);

// rq_tensor.cu: K1 (tcgen05 RQ encode / k-means assignment) and the wide-codebook PQ encode
// The fused k-means pass: the assignment pass also accumulates the rows under their PREVIOUS assignment into per-CTA
// partial sums | counts ([grid][K][d] floats, [grid][K] ints; grid = min(ceil(n / 256), SM count)).
struct KmeansFusedPass {
  const int32_t* prev;
  int64_t prev_stride;
  float* part_sums;
  int32_t* part_counts;
};
bool mevi_rq_tensor_supported(mevi_ctx* ctx, int d, int M, int K, int metric);
bool mevi_kmeans_fused_supported(mevi_ctx* ctx, int d, int K);
// pq_codebook: when non-null, codes are PQ codes of a block-padded `cb` and the rows the prefilter flags are re-decided
// by the sub-vector kernel against this [M][K][d/M] codebook instead of by rq_exact.  km_fused: non-null (M = 1 only)
// runs the fused k-means pass.
int mevi_rq_tensor_assign(mevi_ctx* ctx, const float* X, int64_t n, int d, const float* cb, int M, int K, int metric,
                          int32_t* codes, int64_t codes_stride, float* residual, int64_t* stats, double* inertia,
                          const float* pq_codebook, const KmeansFusedPass* km_fused, cudaStream_t st);
bool mevi_pq_tensor_supported(mevi_ctx* ctx, int64_t n, int d, int M, int K, int metric);
int mevi_pq_tensor_encode(mevi_ctx* ctx, const float* X, int64_t n, int d, const float* cb, int M, int K, int metric,
                          int32_t* codes, cudaStream_t st);

// pq_encode.cu: the fp32 sub-vector kernel as the arbiter of the tensor PQ routes
int mevi_pq_fix_launch(mevi_ctx* ctx, const float* X, int64_t n, int d, const float* pq_codebook, int M, int K, int metric,
                       int32_t* codes, const int32_t* work_rows, const int64_t* n_work_dev, cudaStream_t st);
int mevi_pq_fix_pairs_launch(mevi_ctx* ctx, const float* X, int64_t n, int d, const float* pq_codebook, int M, int K, int metric,
                             int32_t* codes, const uint32_t* pairs, const unsigned long long* n_pairs_dev, unsigned long long cap,
                             const int* overflow, cudaStream_t st);

// flat_tensor.cu: K2 on the tensor cores (*fell_back = 1: the fp32 path has to compute the answer)
bool mevi_flat_tensor_supported(mevi_ctx* ctx, int d, int k);
int mevi_flat_tensor_search(mevi_ctx* ctx, const float* Q, int nq, const float* D, int64_t n, int d, int k,
                            int64_t id_base, float* scores, int64_t* ids, int* fell_back, cudaStream_t st);

#define MEVI_COUNT_LAUNCH(ctx, n) ((ctx)->launches += (n))

#define MEVI_CHECK_CTX(ctx) \
  do {                      \
    if (!(ctx)) return MEVI_ERR_INVALID; \
  } while (0)

#define MEVI_CUDA(ctx, expr)                                                                   \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess)                                                                     \
      return mevi_set_error((ctx), MEVI_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,              \
                            cudaGetErrorString(_e), __FILE__, __LINE__);                      \
  } while (0)

#define MEVI_REQUIRE(ctx, cond, ...)                                        \
  do {                                                                      \
    if (!(cond)) return mevi_set_error((ctx), MEVI_ERR_INVALID, __VA_ARGS__); \
  } while (0)

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
    else prev = -1;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

// ---- device helpers -------------------------------------------------------
__device__ __forceinline__ float4 ldg_f4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

// streaming 128-bit load that does not allocate in L1 (row data read exactly once)
__device__ __forceinline__ float4 ld_stream_f4(const float* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(MEVI_FULL_MASK, v, o);
  return v;
}

// (score desc, id asc) ordering used by every top-k in the library
__device__ __forceinline__ bool topk_before(float sa, int64_t ia, float sb, int64_t ib) {
  return (sa > sb) || (sa == sb && ia < ib);
}

// bitonic sort by a SUBSET of the CTA's warps: threads pass their rank in the group (gtid) and the
// group size; synchronisation uses named barrier `bar_id` (count = nthreads) instead of __syncthreads
template <typename IdT>
__device__ __forceinline__ void group_bitonic_sort(float* s, IdT* id, int n, int gtid, int nthreads, int bar_id) {
  for (int k = 2; k <= n; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = gtid; i < n; i += nthreads) {
        int ixj = i ^ j;
        if (ixj > i) {
          bool up = ((i & k) == 0);
          float a = s[i], b = s[ixj];
          IdT ia = id[i], ib = id[ixj];
          bool a_first = topk_before(a, (int64_t)ia, b, (int64_t)ib);
          if (a_first != up) {
            s[i] = b; s[ixj] = a;
            id[i] = ib; id[ixj] = ia;
          }
        }
      }
      asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "r"(nthreads) : "memory");
    }
  }
}

// ---- radix select over shared-memory floats ------------------------------------------------------------------
// monotone float <-> unsigned key (larger float = larger key)
__device__ __forceinline__ unsigned sel_key(float f) {
  const unsigned u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float sel_unkey(unsigned k) { return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k); }

// The k-th largest (1-based, k <= n) of s[0..n) by a radix select over the bits in which the values differ; every thread
// of a 256-thread CTA calls it and gets the value.  `hist` = 256 unsigned of shared memory, `scratch` = 4 unsigned of
// shared memory; both may be reused afterwards.  Histogram updates are aggregated per warp (equal digits are common).
__device__ __forceinline__ float block256_select_kth(const float* s, int n, int k, unsigned* hist, unsigned* scratch) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) { scratch[0] = 0xFFFFFFFFu; scratch[1] = 0u; }
  __syncthreads();
  unsigned kmin = 0xFFFFFFFFu, kmax = 0u;
  for (int i = tid; i < n; i += 256) {
    const unsigned key = sel_key(s[i]);
    kmin = min(kmin, key);
    kmax = max(kmax, key);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    kmin = min(kmin, __shfl_xor_sync(MEVI_FULL_MASK, kmin, o));
    kmax = max(kmax, __shfl_xor_sync(MEVI_FULL_MASK, kmax, o));
  }
  if (lane == 0) { atomicMin(&scratch[0], kmin); atomicMax(&scratch[1], kmax); }
  __syncthreads();
  const unsigned lo_key = scratch[0], hi_key = scratch[1];
  unsigned prefix = hi_key;
  int rem = k;
  if (lo_key != hi_key) {
    const int top = 31 - __clz(lo_key ^ hi_key);
    int hi_bit = top;
    prefix = (top == 31) ? 0u : (hi_key >> (top + 1)) << (top + 1);
    while (hi_bit >= 0) {
      const int width = hi_bit >= 7 ? 8 : hi_bit + 1;
      const int shift = hi_bit + 1 - width;
      const unsigned above = (hi_bit == 31) ? 0u : (0xFFFFFFFFu << (hi_bit + 1));
      hist[tid] = 0;
      __syncthreads();
      for (int base = 0; base < n; base += 256) {
        const int i = base + tid;
        unsigned digit = 0xFFFFu;
        if (i < n) {
          const unsigned key = sel_key(s[i]);
          if ((key & above) == (prefix & above)) digit = (key >> shift) & ((1u << width) - 1u);
        }
        const unsigned peers = __match_any_sync(MEVI_FULL_MASK, digit);
        if (digit != 0xFFFFu && lane == __ffs(peers) - 1) atomicAdd(&hist[digit], __popc(peers));
      }
      __syncthreads();
      if (warp == 0) {
        int local[8], sum = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) { local[j] = (int)hist[255 - (lane * 8 + j)]; sum += local[j]; }
        int incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int v = __shfl_up_sync(MEVI_FULL_MASK, incl, o);
          if (lane >= o) incl += v;
        }
        const int excl = incl - sum;
        if (excl < rem && rem <= incl) {
          int r = rem - excl;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            if (r > 0 && r <= local[j]) { scratch[2] = 255u - (unsigned)(lane * 8 + j); scratch[3] = (unsigned)r; r = 0; }
            else if (r > 0) r -= local[j];
          }
        }
      }
      __syncthreads();
      prefix |= scratch[2] << shift;
      rem = (int)scratch[3];
      hi_bit = shift - 1;
      __syncthreads();
    }
  }
  return sel_unkey(prefix);
}

// shared-memory bitonic sort of n (power of two) (score,id) pairs into topk_before order
template <typename IdT>
__device__ __forceinline__ void block_bitonic_sort(float* s, IdT* id, int n) {
  for (int k = 2; k <= n; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < n; i += blockDim.x) {
        int ixj = i ^ j;
        if (ixj > i) {
          bool up = ((i & k) == 0);
          float a = s[i], b = s[ixj];
          IdT ia = id[i], ib = id[ixj];
          bool a_first = topk_before(a, (int64_t)ia, b, (int64_t)ib);
          if (a_first != up) {
            s[i] = b; s[ixj] = a;
            id[i] = ib; id[ixj] = ia;
          }
        }
      }
      __syncthreads();
    }
  }
}
