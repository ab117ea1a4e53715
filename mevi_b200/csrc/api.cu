// api.cu — context lifetime, error strings, scratch arenas.
#include <stdarg.h>

#include <stdlib.h>

#include "common.cuh"

int mevi_set_error(mevi_ctx* ctx, int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (ctx) ctx->err = buf;
  return code;
}

void* mevi_ws(mevi_ctx* ctx, int slot, size_t bytes) {
  if (bytes == 0) bytes = 256;
  if (ctx->ws_bytes[slot] >= bytes) return ctx->ws[slot];
  if (ctx->ws[slot]) {
    cudaDeviceSynchronize();
    cudaFree(ctx->ws[slot]);
    ctx->ws[slot] = nullptr;
    ctx->ws_bytes[slot] = 0;
  }
  size_t want = bytes + bytes / 8;  // slack so slowly growing requests do not re-allocate every call
  want = (want + 255) & ~size_t(255);
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, want);
  if (e != cudaSuccess) {
    cudaGetLastError();
    want = (bytes + 255) & ~size_t(255);
    e = cudaMalloc(&p, want);
  }
  if (e != cudaSuccess) {
    cudaGetLastError();
    mevi_set_error(ctx, MEVI_ERR_NOMEM, "cudaMalloc(%zu bytes) for scratch slot %d failed: %s", want, slot,
                   cudaGetErrorString(e));
    return nullptr;
  }
  ctx->ws[slot] = p;
  ctx->ws_bytes[slot] = want;
  return p;
}

void* mevi_pinned(mevi_ctx* ctx, int slot, size_t bytes) {
  if (ctx->pinned_bytes[slot] >= bytes) return ctx->pinned[slot];
  if (ctx->pinned[slot]) {
    cudaFreeHost(ctx->pinned[slot]);
    ctx->pinned[slot] = nullptr;
    ctx->pinned_bytes[slot] = 0;
  }
  void* p = nullptr;
  cudaError_t e = cudaMallocHost(&p, bytes);
  if (e != cudaSuccess) {
    cudaGetLastError();
    mevi_set_error(ctx, MEVI_ERR_NOMEM, "cudaMallocHost(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
    return nullptr;
  }
  ctx->pinned[slot] = p;
  ctx->pinned_bytes[slot] = bytes;
  return p;
}

int mevi_publish_errors(mevi_ctx* ctx, cudaStream_t st) {
  MEVI_CUDA(ctx, cudaMemcpyAsync((void*)ctx->host_err, ctx->dev_err, MEVI_ERRSLOTS * sizeof(int), cudaMemcpyDeviceToHost, st));
  return MEVI_OK;
}

int mevi_deferred_error(mevi_ctx* ctx) {
  static const char* const who[MEVI_ERRSLOTS] = {"tensor RQ encode", "cluster re-rank", "kernel", "kernel", "kernel", "kernel", "kernel", "kernel"};
  for (int i = 0; i < MEVI_ERRSLOTS; ++i) {
    const int code = ctx->host_err[i];
    if (code != 0) {
      for (int j = 0; j < MEVI_ERRSLOTS; ++j) ctx->host_err[j] = 0;
      cudaMemset(ctx->dev_err, 0, MEVI_ERRSLOTS * sizeof(int));
      return mevi_set_error(ctx, MEVI_ERR_CUDA,
                            "%s: a pipeline wait timed out on the device (code %d); the results of that launch are invalid "
                            "(codes were overwritten with -1, top-k lists are incomplete)", who[i], code);
    }
  }
  return MEVI_OK;
}

extern "C" {

int mevi_abi_version(void) { return MEVI_ABI_VERSION; }

int mevi_ctx_check(mevi_ctx* ctx, void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  MEVI_CUDA(ctx, cudaStreamSynchronize((cudaStream_t)stream));
  return mevi_deferred_error(ctx);
}

int mevi_ctx_create(int device, mevi_ctx** out) {
  if (!out) return MEVI_ERR_INVALID;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) {
    cudaGetLastError();
    return MEVI_ERR_CUDA;
  }
  mevi_ctx* ctx = new mevi_ctx();
  ctx->device = device;
  DeviceGuard g(device);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) {
    delete ctx;
    return MEVI_ERR_CUDA;
  }
  ctx->sm_count = prop.multiProcessorCount;
  ctx->cc_major = prop.major;
  ctx->cc_minor = prop.minor;
  ctx->total_mem = prop.totalGlobalMem;
  ctx->l2_bytes = (size_t)prop.l2CacheSize;
  for (int i = 0; i < 2; ++i) cudaStreamCreateWithFlags(&ctx->aux_stream[i], cudaStreamNonBlocking);
  for (int i = 0; i < 4; ++i) cudaEventCreateWithFlags(&ctx->aux_event[i], cudaEventDisableTiming);
  int* herr = nullptr;
  if (cudaMalloc(&ctx->dev_err, MEVI_ERRSLOTS * sizeof(int)) != cudaSuccess ||
      cudaMallocHost(&herr, MEVI_ERRSLOTS * sizeof(int)) != cudaSuccess) {
    cudaGetLastError();
    mevi_ctx_destroy(ctx);
    return MEVI_ERR_NOMEM;
  }
  ctx->host_err = herr;
  cudaMemset(ctx->dev_err, 0, MEVI_ERRSLOTS * sizeof(int));
  for (int i = 0; i < MEVI_ERRSLOTS; ++i) ctx->host_err[i] = 0;
  *out = ctx;
  return MEVI_OK;
}

void mevi_ctx_destroy(mevi_ctx* ctx) {
  if (!ctx) return;
  DeviceGuard g(ctx->device);
  cudaDeviceSynchronize();
  for (int i = 0; i < WS_NUM; ++i)
    if (ctx->ws[i]) cudaFree(ctx->ws[i]);
  for (int i = 0; i < 4; ++i)
    if (ctx->pinned[i]) cudaFreeHost(ctx->pinned[i]);
  if (ctx->dev_err) cudaFree(ctx->dev_err);
  if (ctx->host_err) cudaFreeHost((void*)ctx->host_err);
  for (int i = 0; i < 2; ++i)
    if (ctx->aux_stream[i]) cudaStreamDestroy(ctx->aux_stream[i]);
  for (int i = 0; i < 4; ++i)
    if (ctx->aux_event[i]) cudaEventDestroy(ctx->aux_event[i]);
  free(ctx->gr_plan);
  free(ctx->gr_mc);
  delete ctx;
}

const char* mevi_last_error(mevi_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int mevi_device_info(mevi_ctx* ctx, int64_t info[8]) {
  MEVI_CHECK_CTX(ctx);
  if (!info) return mevi_set_error(ctx, MEVI_ERR_INVALID, "info is NULL");
  info[0] = ctx->sm_count;
  info[1] = ctx->cc_major;
  info[2] = ctx->cc_minor;
  info[3] = (int64_t)ctx->total_mem;
  info[4] = (ctx->cc_major == 10) ? 1 : 0;
  info[5] = (int64_t)ctx->l2_bytes;
  info[6] = ctx->launches;
  info[7] = 0;
  return MEVI_OK;
}

}  // extern "C"
