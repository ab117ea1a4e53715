// rq_api.cu — C-ABI entry points of the RQ encode (device- and host-buffer forms).
#include "common.cuh"

namespace {
__global__ void stats_add_kernel(int64_t* stats, int64_t flagged, int64_t rows) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    atomicAdd((unsigned long long*)&stats[0], (unsigned long long)flagged);
    atomicAdd((unsigned long long*)&stats[1], (unsigned long long)rows);
  }
}

int encode_dispatch(mevi_ctx* ctx, const float* X, int64_t n, int d, const float* cb, int M, int K, int metric, int mode,
                    int32_t* codes, float* residual, int64_t* stats_accum, cudaStream_t st) {
  bool use_tensor = false;
  if (mode == MEVI_MODE_TENSOR) {
    if (!mevi_rq_tensor_supported(ctx, d, M, K, metric))
      return mevi_set_error(ctx, MEVI_ERR_UNSUPPORTED,
                            "tensor RQ encode unsupported for d=%d M=%d K=%d metric=%d on cc %d.%d", d, M, K, metric,
                            ctx->cc_major, ctx->cc_minor);
    use_tensor = true;
  } else if (mode == MEVI_MODE_AUTO) {
    use_tensor = mevi_rq_tensor_supported(ctx, d, M, K, metric) && n >= 4096;
  } else if (mode != MEVI_MODE_EXACT) {
    return mevi_set_error(ctx, MEVI_ERR_INVALID, "unknown mode %d", mode);
  }
  if (use_tensor)
    return mevi_rq_tensor_assign(ctx, X, n, d, cb, M, K, metric, codes, M, residual, stats_accum, nullptr, nullptr, nullptr, st);
  int rc = mevi_rq_exact_launch(ctx, X, n, d, cb, M, K, metric, codes, M, residual, nullptr, nullptr, nullptr, n, nullptr, st);
  if (rc != MEVI_OK) return rc;
  if (stats_accum) {
    stats_add_kernel<<<1, 32, 0, st>>>(stats_accum, 0, n);
    MEVI_COUNT_LAUNCH(ctx, 1);
    MEVI_CUDA(ctx, cudaGetLastError());
  }
  return MEVI_OK;
}
}  // namespace

extern "C" {

int mevi_rq_encode(mevi_ctx* ctx, const float* X, int64_t n, int d, const float* codebook, int M, int K, int metric,
                   int mode, int32_t* codes, float* residual_or_null, int64_t* stats_or_null, void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  MEVI_REQUIRE(ctx, n >= 0 && n < (int64_t)2147483647, "n out of range");
  MEVI_REQUIRE(ctx, codebook && ((codes && X) || n == 0), "NULL argument");
  MEVI_REQUIRE(ctx, metric == MEVI_METRIC_L2 || metric == MEVI_METRIC_IP, "unknown metric %d", metric);
  if (stats_or_null) MEVI_CUDA(ctx, cudaMemsetAsync(stats_or_null, 0, 8 * sizeof(int64_t), st));
  if (n == 0) return MEVI_OK;
  return encode_dispatch(ctx, X, n, d, codebook, M, K, metric, mode, codes, residual_or_null, stats_or_null, st);
}

int mevi_rq_encode_host(mevi_ctx* ctx, const float* X_host, int64_t n, int d, const float* codebook_host, int M, int K,
                        int metric, int mode, int32_t* codes_host, int64_t chunk_rows, int64_t* stats_host_or_null) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  MEVI_REQUIRE(ctx, codebook_host && codes_host && (X_host || n == 0), "NULL argument");
  MEVI_REQUIRE(ctx, n >= 0 && d > 0 && M >= 1 && K >= 1, "bad shape");
  if (chunk_rows <= 0) chunk_rows = (int64_t)1 << 18;  // 262,144 rows = 805 MB at d=768
  if (chunk_rows > n && n > 0) chunk_rows = n;
  const size_t cb_bytes = (size_t)M * K * d * sizeof(float);
  char* misc = (char*)mevi_ws(ctx, WS_MISC, cb_bytes + 64);
  if (!misc) return MEVI_ERR_NOMEM;
  float* cb_dev = (float*)misc;
  int64_t* stats_dev = (int64_t*)(misc + ((cb_bytes + 63) & ~size_t(63)));
  // (stats_dev needs 64 bytes past the aligned codebook)
  if (ctx->ws_bytes[WS_MISC] < ((cb_bytes + 63) & ~size_t(63)) + 64) {
    misc = (char*)mevi_ws(ctx, WS_MISC, cb_bytes + 256);
    if (!misc) return MEVI_ERR_NOMEM;
    cb_dev = (float*)misc;
    stats_dev = (int64_t*)(misc + ((cb_bytes + 63) & ~size_t(63)));
  }
  cudaStream_t s_copy = ctx->aux_stream[0], s_comp = ctx->aux_stream[1];
  MEVI_CUDA(ctx, cudaMemcpyAsync(cb_dev, codebook_host, cb_bytes, cudaMemcpyHostToDevice, s_comp));
  MEVI_CUDA(ctx, cudaMemsetAsync(stats_dev, 0, 8 * sizeof(int64_t), s_comp));
  if (n > 0) {
    float* stage[2];
    int32_t* cdev[2];
    stage[0] = (float*)mevi_ws(ctx, WS_HOST_STAGE_A, (size_t)chunk_rows * d * sizeof(float));
    stage[1] = (float*)mevi_ws(ctx, WS_HOST_STAGE_B, (size_t)chunk_rows * d * sizeof(float));
    cdev[0] = (int32_t*)mevi_ws(ctx, WS_HOST_CODES_A, (size_t)chunk_rows * M * sizeof(int32_t));
    cdev[1] = (int32_t*)mevi_ws(ctx, WS_HOST_CODES_B, (size_t)chunk_rows * M * sizeof(int32_t));
    if (!stage[0] || !stage[1] || !cdev[0] || !cdev[1]) return MEVI_ERR_NOMEM;
    cudaEvent_t h2d_done[2] = {ctx->aux_event[0], ctx->aux_event[1]};
    cudaEvent_t comp_done[2] = {ctx->aux_event[2], ctx->aux_event[3]};
    int64_t ci = 0;
    for (int64_t off = 0; off < n; off += chunk_rows, ++ci) {
      const int b = (int)(ci & 1);
      const int64_t rows = (n - off) < chunk_rows ? (n - off) : chunk_rows;
      if (ci >= 2) MEVI_CUDA(ctx, cudaStreamWaitEvent(s_copy, comp_done[b], 0));
      MEVI_CUDA(ctx, cudaMemcpyAsync(stage[b], X_host + off * d, (size_t)rows * d * sizeof(float),
                                     cudaMemcpyHostToDevice, s_copy));
      MEVI_CUDA(ctx, cudaEventRecord(h2d_done[b], s_copy));
      MEVI_CUDA(ctx, cudaStreamWaitEvent(s_comp, h2d_done[b], 0));
      int rc = encode_dispatch(ctx, stage[b], rows, d, cb_dev, M, K, metric, mode, cdev[b], nullptr, stats_dev, s_comp);
      if (rc != MEVI_OK) {
        cudaStreamSynchronize(s_copy);
        cudaStreamSynchronize(s_comp);
        return rc;
      }
      MEVI_CUDA(ctx, cudaMemcpyAsync(codes_host + off * M, cdev[b], (size_t)rows * M * sizeof(int32_t),
                                     cudaMemcpyDeviceToHost, s_comp));
      MEVI_CUDA(ctx, cudaEventRecord(comp_done[b], s_comp));
    }
  }
  if (stats_host_or_null)
    MEVI_CUDA(ctx, cudaMemcpyAsync(stats_host_or_null, stats_dev, 8 * sizeof(int64_t), cudaMemcpyDeviceToHost, s_comp));
  MEVI_CUDA(ctx, cudaStreamSynchronize(s_copy));
  MEVI_CUDA(ctx, cudaStreamSynchronize(s_comp));
  return mevi_deferred_error(ctx);  // a pipeline time-out in any chunk's kernel fails the call
}

}  // extern "C"
