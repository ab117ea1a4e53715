// invlists.cu — inverted-list (leaf -> doc ids) construction on the device.
// Replaces the python dict loops of MEVI/pq.py:236-242 and 200-214: the leaf key
// of a row is its code tuple read as a base-K number; a stable radix sort of
// (key, row) pairs gives, per leaf, the doc ids in ascending order — exactly the
// append order of the reference's defaultdict(list).
#include <cub/cub.cuh>

#include "common.cuh"

namespace {
__global__ void leaf_key_kernel(const int32_t* __restrict__ codes, int64_t n, int M, int K, int64_t* __restrict__ keys,
                                int32_t* __restrict__ rows) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t key = 0;
    for (int j = 0; j < M; ++j) key = key * K + codes[i * M + j];
    keys[i] = key;
    rows[i] = (int32_t)i;
  }
}

// beam-search leaves (code tuples) -> index of the leaf in the sorted key list, -1 when no document lives there
// (`doc_cluster.get(tuple, None)`, main_models.py:3928) or a code is outside [0, K)
__global__ void leaf_lookup_kernel(const int64_t* __restrict__ dec, int64_t n_pairs, int M, int K,
                                   const int64_t* __restrict__ leaf_keys, int64_t n_leaves, int32_t* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_pairs) return;
  int64_t key = 0;
  bool valid = true;
  for (int j = 0; j < M; ++j) {
    const int64_t c = dec[i * M + j];
    valid &= (c >= 0) && (c < K);
    key = key * K + c;
  }
  int32_t r = -1;
  if (valid && n_leaves > 0) {
    int64_t lo = 0, hi = n_leaves;  // lower bound
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (leaf_keys[mid] < key) lo = mid + 1; else hi = mid;
    }
    if (lo < n_leaves && leaf_keys[lo] == key) r = (int32_t)lo;
  }
  out[i] = r;
}

__global__ void occ_pairs_kernel(const int32_t* __restrict__ docids, int64_t n, int32_t* __restrict__ keys,
                                 int32_t* __restrict__ pos) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    keys[i] = docids[i];
    pos[i] = (int32_t)i;
  }
}

__device__ __forceinline__ int32_t leaf_of_position(const int64_t* __restrict__ off, int64_t n_leaves, int64_t p) {
  int64_t lo = 0, hi = n_leaves;  // last leaf whose first position is <= p
  while (hi - lo > 1) {
    const int64_t mid = (lo + hi) >> 1;
    if (off[mid] <= p) lo = mid; else hi = mid;
  }
  return (int32_t)lo;
}

// one thread per group head of the (document, position)-sorted pairs: the group is the document's positions, ascending
// (stable sort of ascending positions).  Counts the group (max_occ) and with occ != NULL writes every member's row.
__global__ void occ_groups_kernel(const int32_t* __restrict__ keys, const int32_t* __restrict__ pos, int64_t n,
                                  const int64_t* __restrict__ off, int64_t n_leaves, int width, int32_t* __restrict__ occ,
                                  int* __restrict__ max_occ) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    if (i > 0 && keys[i - 1] == keys[i]) continue;
    int64_t j = i + 1;
    while (j < n && keys[j] == keys[i]) ++j;
    const int64_t size = j - i;
    atomicMax(max_occ, (int)(size < 0x7fffffff ? size : 0x7fffffff));
    if (!occ || size - 1 > width) continue;
    for (int64_t a = i; a < j; ++a) {
      const int32_t own = leaf_of_position(off, n_leaves, pos[a]);
      int32_t* row = occ + (int64_t)pos[a] * width;
      int w = 0;
      for (int64_t b = i; b < j; ++b) {
        if (b == a) continue;
        const int32_t leaf = leaf_of_position(off, n_leaves, pos[b]);
        row[w++] = (leaf == own && b < a) ? -2 - leaf : leaf;  // an earlier position of the same leaf: -2 - leaf
      }
      for (; w < width; ++w) row[w] = -1;
    }
  }
}
}  // namespace

extern "C" int mevi_occurrence_table(mevi_ctx* ctx, const int64_t* leaf_offsets, int64_t n_leaves, const int32_t* leaf_docids,
                                     int64_t n, int width, int32_t* occ_leaves, int32_t* max_occ_host, void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  MEVI_REQUIRE(ctx, leaf_offsets && max_occ_host && (leaf_docids || n == 0), "NULL argument");
  MEVI_REQUIRE(ctx, n >= 0 && n < (int64_t)2147483647 && n_leaves >= 0 && width >= 0, "bad shape");
  *max_occ_host = 0;
  if (n == 0) return MEVI_OK;
  const size_t arr = ((size_t)n * sizeof(int32_t) + 255) & ~size_t(255);
  char* ws = (char*)mevi_ws(ctx, WS_SORT_KEYS, 4 * arr + 256);
  if (!ws) return MEVI_ERR_NOMEM;
  int32_t* keys_in = (int32_t*)ws;
  int32_t* pos_in = (int32_t*)(ws + arr);
  int32_t* keys = (int32_t*)(ws + 2 * arr);
  int32_t* pos = (int32_t*)(ws + 3 * arr);
  int* d_max = (int*)(ws + 4 * arr);
  int h_max = 0;
  const int grid = ctx->sm_count * 8;
  occ_pairs_kernel<<<grid, 256, 0, st>>>(leaf_docids, n, keys_in, pos_in);
  MEVI_COUNT_LAUNCH(ctx, 1);
  MEVI_CUDA(ctx, cudaGetLastError());
  size_t tmp_bytes = 0;
  MEVI_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, keys_in, keys, pos_in, pos, (int)n, 0, 31, st));
  void* tmp = mevi_ws(ctx, WS_SORT_TMP, tmp_bytes);
  if (!tmp) return MEVI_ERR_NOMEM;
  MEVI_CUDA(ctx, cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, keys_in, keys, pos_in, pos, (int)n, 0, 31, st));
  for (int pass = 0; pass < 2; ++pass) {  // pass 0 counts; pass 1 writes once the width is known to suffice
    MEVI_CUDA(ctx, cudaMemsetAsync(d_max, 0, sizeof(int), st));
    occ_groups_kernel<<<grid, 256, 0, st>>>(keys, pos, n, leaf_offsets, n_leaves, width, pass ? occ_leaves : nullptr, d_max);
    MEVI_COUNT_LAUNCH(ctx, 1);
    MEVI_CUDA(ctx, cudaGetLastError());
    MEVI_CUDA(ctx, cudaMemcpyAsync(&h_max, d_max, sizeof(int), cudaMemcpyDeviceToHost, st));
    MEVI_CUDA(ctx, cudaStreamSynchronize(st));
    *max_occ_host = h_max;
    if (!occ_leaves) break;
    MEVI_REQUIRE(ctx, width >= h_max - 1, "occurrence table width %d < C - 1 = %d", width, h_max - 1);
  }
  return MEVI_OK;
}

extern "C" int mevi_leaf_lookup(mevi_ctx* ctx, const int64_t* leaves, int64_t n_pairs, int M, int K,
                                const int64_t* leaf_keys, int64_t n_leaves, int32_t* leaf_index, void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  MEVI_REQUIRE(ctx, leaves && leaf_index && (leaf_keys || n_leaves == 0), "NULL argument");
  MEVI_REQUIRE(ctx, M >= 1 && K >= 1 && n_leaves >= 0 && n_leaves < (int64_t)2147483647, "bad shape");
  if (n_pairs <= 0) return MEVI_OK;
  leaf_lookup_kernel<<<(unsigned)((n_pairs + 255) / 256), 256, 0, (cudaStream_t)stream>>>(leaves, n_pairs, M, K, leaf_keys,
                                                                                           n_leaves, leaf_index);
  MEVI_CUDA(ctx, cudaGetLastError());
  MEVI_COUNT_LAUNCH(ctx, 1);
  return MEVI_OK;
}

extern "C" int mevi_build_inverted_lists(mevi_ctx* ctx, const int32_t* codes, int64_t n, int M, int K,
                                         int32_t* sorted_docids, int64_t* sorted_keys, void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  MEVI_REQUIRE(ctx, codes && sorted_docids && sorted_keys, "NULL argument");
  MEVI_REQUIRE(ctx, n >= 0 && n < (int64_t)2147483647 && M >= 1 && K >= 1, "bad shape");
  double bits = 0;
  for (int j = 0; j < M; ++j) bits += log2((double)K);
  MEVI_REQUIRE(ctx, bits < 62.0, "K^M does not fit a 62-bit leaf key");
  if (n == 0) return MEVI_OK;
  int end_bit = (int)ceil(bits);
  if (end_bit < 1) end_bit = 1;
  char* in = (char*)mevi_ws(ctx, WS_SORT_KEYS, (size_t)n * (sizeof(int64_t) + sizeof(int32_t)) + 256);
  if (!in) return MEVI_ERR_NOMEM;
  int64_t* keys_in = (int64_t*)in;
  int32_t* rows_in = (int32_t*)(in + (((size_t)n * sizeof(int64_t) + 255) & ~size_t(255)));
  if (ctx->ws_bytes[WS_SORT_KEYS] < (((size_t)n * sizeof(int64_t) + 255) & ~size_t(255)) + (size_t)n * sizeof(int32_t)) {
    in = (char*)mevi_ws(ctx, WS_SORT_KEYS, (size_t)n * 12 + 1024);
    if (!in) return MEVI_ERR_NOMEM;
    keys_in = (int64_t*)in;
    rows_in = (int32_t*)(in + (((size_t)n * sizeof(int64_t) + 255) & ~size_t(255)));
  }
  int grid = ctx->sm_count * 8;
  leaf_key_kernel<<<grid, 256, 0, st>>>(codes, n, M, K, keys_in, rows_in);
  MEVI_COUNT_LAUNCH(ctx, 1);
  MEVI_CUDA(ctx, cudaGetLastError());
  size_t tmp_bytes = 0;
  MEVI_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, keys_in, sorted_keys, rows_in, sorted_docids,
                                                 (int)n, 0, end_bit, st));
  void* tmp = mevi_ws(ctx, WS_SORT_TMP, tmp_bytes);
  if (!tmp) return MEVI_ERR_NOMEM;
  MEVI_CUDA(ctx, cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, keys_in, sorted_keys, rows_in, sorted_docids, (int)n, 0,
                                                 end_bit, st));
  return MEVI_OK;
}
