// flat_tensor.cu — K2: exact flat inner-product top-k with a tcgen05 fp16 prefilter.
//
// Replaces MEVI/faiss_search.py:13-21 with param='Flat' (faiss IndexFlatIP add + search) for large
// inputs.  The dense contraction Q[nq,d].D[N,d]^T runs on the 5th-generation tensor cores in fp16
// (one pass, fp32 accumulation in TMEM); because fp16 rounding perturbs a score by at most
//     E(q,d) = 1.01 * 2^-10 * |q| * |d|            (two RN roundings to 11 bits per product)
// the tensor result is only a PREFILTER: a document is kept for a query if its approximate score is
// within 2*E_max of the query's running k-th best approximate score, which provably includes every
// member of the exact top-k; the survivors (k plus a few dozen) are re-scored in exact fp32 and sorted.
// If more survivors than the buffer holds fall inside the margin, the call falls back to the fp32
// CUDA-core search of flat_ip.cu, so the answer is always the exact one.
//
// Data path.  One streaming pass converts D (and Q) to fp16 "images": [tile][K chunk][rows][64 halfs]
// with the 128-byte XOR swizzle UMMA expects, so every pipeline stage is ONE contiguous block fetched
// by a single bulk async copy (no tensor maps).  GEMM CTA (persistent, 320 threads): warp 0 = bulk-copy
// producer (A: 128 docs x 64, 16 KB; B: 256 queries x 64, 32 KB; 4 stages), warp 1 = one thread issuing
// tcgen05.mma M=128 N=256 K=16, accumulators double-buffered in TMEM (2 x 256 columns), warps 2-5 =
// epilogue: tcgen05.ld, compare with the per-query threshold, rare atomic append.  Work items are
// (doc tile, query block) pairs in doc-tile-major order so a doc tile is reused from L2 by all query
// blocks.  Roofline: tensor pipe (2*nq*N*d FLOP); L2->SM operand traffic is the practical limiter.
#include <cuda_fp16.h>
#include <math_constants.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "ptx.cuh"

namespace {

constexpr int FT_TM = 128;       // docs per tile (UMMA M)
constexpr int FT_TN = 256;       // queries per block (UMMA N)
constexpr int FT_KC = 64;        // K elements per chunk (128-byte rows)
constexpr int FT_STAGES = 4;
constexpr int FT_A_BYTES = FT_TM * 128, FT_B_BYTES = FT_TN * 128;
constexpr int FT_STAGE_BYTES = FT_A_BYTES + FT_B_BYTES;  // 48 KB
constexpr int FT_EPI_WARPS = 8;   // two per TMEM lane group, 128 of the 256 accumulator columns each
constexpr int FT_THREADS2 = 64 + 32 * FT_EPI_WARPS;
constexpr int FT_DEFAULT_CLUSTER = 2;
constexpr int FT_KEEP = 512;     // approximate candidates kept per query between chunks

enum { FC_SD = 0, FC_SQ, FC_INV, FC_DMAX, FC_CLAMPED, FC_NUM = 8 };

// ---- fp32 -> swizzled fp16 image, one warp per row; also row norms and the maximum norm -----------
__global__ void to_fp16_image_kernel(const float* __restrict__ X, int64_t rows, int d, int rows_per_tile,
                                     const float* __restrict__ consts, int scale_slot, __half* __restrict__ img,
                                     float* __restrict__ norms, unsigned* __restrict__ max_norm_bits,
                                     int* __restrict__ clamped, int64_t padded_rows,
                                     const int32_t* __restrict__ src_index = nullptr) {  // image row -> row of X, -1 = zero row
  const int lane = threadIdx.x & 31;
  const int64_t warp_global = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const float s = consts[scale_slot];
  const int units = d / 8;  // 16-byte units per row
  const int nchunks = d / FT_KC;
  for (int64_t prow = warp_global; prow < padded_rows; prow += n_warps) {
    const int64_t tile = prow / rows_per_tile;
    const int r = (int)(prow - tile * rows_per_tile);
    // `row` is the source row; without an index it is the image row itself (rows past the end are zero-filled)
    const int64_t row = src_index ? (src_index[prow] >= 0 ? (int64_t)src_index[prow] : rows) : prow;
    float nrm = 0.f;
    bool clamp = false;
    // four 32-byte units per lane in flight before anything is converted (d = 768 -> the whole row in one round)
    for (int u0 = lane; u0 < units; u0 += 128) {
      float4 va[4], vb[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int u = u0 + 32 * i;
        if (u < units && row < rows) {
          va[i] = ld_stream_f4(X + row * d + u * 8);
          vb[i] = ld_stream_f4(X + row * d + u * 8 + 4);
        } else {
          va[i] = make_float4(0.f, 0.f, 0.f, 0.f);
          vb[i] = va[i];
        }
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int u = u0 + 32 * i;
        if (u >= units) break;
        const float v[8] = {va[i].x, va[i].y, va[i].z, va[i].w, vb[i].x, vb[i].y, vb[i].z, vb[i].w};
        __half h[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          nrm = fmaf(v[e], v[e], nrm);
          float t = v[e] * s;
          if (fabsf(t) > 65000.f) { t = copysignf(65000.f, t); clamp = true; }
          h[e] = __float2half_rn(t);
        }
        const int chunk = u / 8, uu = u & 7;
        __half* dst = img + (((size_t)tile * nchunks + chunk) * rows_per_tile + r) * FT_KC + ((uu ^ (r & 7)) * 8);
        *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(h);
      }
    }
    nrm = warp_sum(nrm);
    if (lane == 0 && row < rows) {
      const float nn = sqrtf(nrm);
      if (norms) norms[row] = nn;
      // one address for every row: test with a plain load first so the atomic fires a handful of times, not N times
      if (max_norm_bits && __float_as_uint(nn) > *(volatile unsigned*)max_norm_bits) atomicMax(max_norm_bits, __float_as_uint(nn));
    }
    if (clamp) atomicExch(clamped, 1);
  }
}

__global__ void flat_absmax_kernel(const float* __restrict__ p, int64_t rows, int d, int64_t row_step, unsigned* out) {
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

// Document-side metadata of a flat search (device, 4 words): [0] sampled |D|max bits, [1] scale 2^s as float,
// [2] largest document norm bits, [3] 1 if a scaled element left the fp16 range.  Written once per image
// (mevi_flat_index_create, or per call in the one-shot search).
enum { DM_ABSMAX = 0, DM_SCALE, DM_MAXNORM, DM_CLAMPED, DM_NUM = 4 };

__global__ void flat_doc_scale_kernel(unsigned* docmeta) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    // 2^s with absmax * 2^s in [2^11, 2^12): 16x headroom below the fp16 maximum (D is only sampled)
    const float ad = __uint_as_float(docmeta[DM_ABSMAX]);
    reinterpret_cast<float*>(docmeta)[DM_SCALE] = ad > 0.f ? ldexpf(1.f, 11 - ilogbf(ad)) : 1.f;
  }
}

// grouped re-rank: scales from [0] the image's |D|max bits and [1] the call's |Q|max bits
__global__ void gr_consts_kernel(const unsigned* absmax2, float* consts) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    const float ad = __uint_as_float(absmax2[0]), aq = __uint_as_float(absmax2[1]);
    const float sd = ad > 0.f ? ldexpf(1.f, 11 - ilogbf(ad)) : 1.f;
    const float sq = aq > 0.f ? ldexpf(1.f, 11 - ilogbf(aq)) : 1.f;
    consts[FC_SD] = sd;
    consts[FC_SQ] = sq;
    consts[FC_INV] = 1.f / (sd * sq);
  }
}

__global__ void flat_consts_kernel(const unsigned* docmeta, const unsigned* absmax_q, float* consts) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    const float sd = reinterpret_cast<const float*>(docmeta)[DM_SCALE], aq = __uint_as_float(absmax_q[0]);
    const float sq = aq > 0.f ? ldexpf(1.f, 11 - ilogbf(aq)) : 1.f;
    consts[FC_SD] = sd;
    consts[FC_SQ] = sq;
    consts[FC_INV] = 1.f / (sd * sq);
  }
}

// per-query slack: a true top-k member's approximate score is at least (k-th approximate) - 2 E_max, with
//   E_max = (1.01 * 2^-10 + d * 2^-23) |q| dmax  +  1.01 * sqrt(d) * 2^-25 * (dmax / sq + |q| / sd)
// The first term is the relative rounding of both fp16 images (2^-11 each) plus the fp32 accumulation of d products
// inside the MMA (d * 2^-23 of sum |q_j d_j|: the worst case of d additions, even if the tensor core truncates; the 1%
// slack alone would not cover it, 2^-16.6 against up to 2^-12 at d = 4096).  The second is the fp16 underflow floor:
// the scales sq, sd are one power of two per call / per image, so the elements of a query whose norm is far below the
// batch's largest become subnormals or zeros, each off by up to 2^-25 / sq absolutely (2^-25 / sd for documents).
__global__ void flat_margin_kernel(const float* __restrict__ qnorm, int nq, int d, const unsigned* __restrict__ dmax_bits,
                                   const float* __restrict__ consts, float* __restrict__ margin) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nq) {
    const float dmax = __uint_as_float(*dmax_bits), qn = qnorm[i];
    const float rel = (1.01f * 9.765625e-4f + (float)d * 1.1920929e-7f) * qn * dmax;
    const float floor_abs = 1.01f * sqrtf((float)d) * 2.9802322e-8f * (dmax / consts[FC_SQ] + qn / consts[FC_SD]);
    margin[i] = 2.f * (rel + floor_abs);
  }
}

struct GemmParams {
  const __half* Aimg; const __half* Bimg;
  int64_t tile_begin, tile_end;   // doc tiles of this chunk
  int64_t n_end;                  // first invalid doc row
  int nq, n_qblocks, nchunks;
  int qparts;                     // query-block range of a tile group split into this many work items
  const float* consts; const float* tau; const float* margin;
  int* count; float* cand_score; int32_t* cand_id; int* overflow; int capg;
  int* err_flag;
};

// CS = CTAs per cluster.  The CS CTAs of a cluster work on CS consecutive doc tiles against the SAME query
// block: each CTA fetches its own A tile and 1/CS of the B block, the latter multicast into every CTA of the
// cluster, so the L2 serves (16 + 32/CS) KB per CTA and stage instead of 48 KB (the L2 slice output, ~6300
// B/clk chip-wide, is what bounds the single-CTA form).  The CTAs therefore advance stage by stage together:
// a stage's empty barrier collects one tcgen05.commit from every CTA of the cluster.
template <int CS>
__global__ void __launch_bounds__(FT_THREADS2, 1) flat_gemm_kernel(GemmParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* ring = smem;  // [FT_STAGES][A 16 KB | B 32 KB]
  float* s_thr = reinterpret_cast<float*>(smem + (size_t)FT_STAGES * FT_STAGE_BYTES);  // [2][FT_TN]
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_thr + 2 * FT_TN);
  uint64_t* full = bars;
  uint64_t* empty = full + FT_STAGES;
  uint64_t* acc_full = empty + FT_STAGES;
  uint64_t* acc_empty = acc_full + 2;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(acc_empty + 2);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < FT_STAGES; ++s) { ptx::mbar_init(&full[s], 1); ptx::mbar_init(&empty[s], CS); }
    for (int b = 0; b < 2; ++b) { ptx::mbar_init(&acc_full[b], 1); ptx::mbar_init(&acc_empty[b], FT_EPI_WARPS); }
    ptx::mbar_fence_init();
  }
  if (warp == 0) ptx::tmem_alloc(tmem_holder, 512);
  ptx::tc_fence_before_sync();
  __syncthreads();
  if (CS > 1) ptx::cluster_sync_all();  // peers' barriers are initialised before anything is multicast at them
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_holder;

  const uint32_t crank = CS > 1 ? ptx::cluster_ctarank() : 0u;
  const int64_t cluster_id = blockIdx.x / CS, n_clusters = gridDim.x / CS;
  constexpr uint16_t CMASK = (uint16_t)((1u << CS) - 1u);
  constexpr int B_SLICE = FT_B_BYTES / CS;
  // Work item = (group of CS doc tiles, part of the query-block range).  A cluster keeps ITS doc tiles for a whole
  // run of query blocks (first use from HBM, the rest from L2) and starts the run at a cluster-dependent block, so
  // at any moment the CTAs of the grid ask the L2 for different A tiles and different B blocks.  (Doc-tile-major
  // order over the whole grid had 28 CTAs miss on the same new A tile at the same moment: 19x the A bytes from HBM.)
  const int64_t n_groups = (p.tile_end - p.tile_begin + CS - 1) / CS;
  const int64_t n_items = n_groups * p.qparts;
  const int nchunks = p.nchunks;
  auto item_range = [&](int64_t w, int64_t& grp, int& qb0, int& len) {
    grp = w / p.qparts;
    const int part = (int)(w % p.qparts);
    qb0 = (int)((int64_t)part * p.n_qblocks / p.qparts);
    len = (int)((int64_t)(part + 1) * p.n_qblocks / p.qparts) - qb0;
  };
  const int stagger = (int)(cluster_id % 61);

  if (warp == 0) {
    if (lane == 0) {
      uint32_t g = 0;
      bool ok = true;
      for (int64_t w = cluster_id; w < n_items && ok; w += n_clusters) {
        int64_t grp; int qb0, len;
        item_range(w, grp, qb0, len);
        int64_t tile = p.tile_begin + grp * CS + crank;
        if (tile >= p.tile_end) tile = p.tile_end - 1;  // ragged last group: keep the pipeline in step, epilogue skips it
        const __half* a_src = p.Aimg + (size_t)tile * nchunks * FT_TM * FT_KC;
        for (int k = 0; k < len && ok; ++k) {
          const int qb = qb0 + (k + stagger) % len;
          const __half* b_src = p.Bimg + (size_t)qb * nchunks * FT_TN * FT_KC;
          for (int c = 0; c < nchunks; ++c, ++g) {
            const uint32_t s = g % FT_STAGES, ph = (g / FT_STAGES) & 1;
            if (!ptx::mbar_wait_backoff(&empty[s], ph ^ 1, 32)) { atomicExch(p.err_flag, 1); ok = false; break; }
            ptx::mbar_arrive_expect_tx(&full[s], FT_STAGE_BYTES);
            uint8_t* st_a = ring + (size_t)s * FT_STAGE_BYTES;
            ptx::bulk_g2s(st_a, a_src + (size_t)c * FT_TM * FT_KC, FT_A_BYTES, &full[s]);
            if (CS == 1) {
              ptx::bulk_g2s(st_a + FT_A_BYTES, b_src + (size_t)c * FT_TN * FT_KC, FT_B_BYTES, &full[s]);
            } else {
              ptx::bulk_g2s_multicast(st_a + FT_A_BYTES + crank * B_SLICE,
                                      reinterpret_cast<const uint8_t*>(b_src + (size_t)c * FT_TN * FT_KC) + crank * B_SLICE, B_SLICE,
                                      &full[s], CMASK);
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = ptx::umma_idesc_f16_m128(FT_TN);
      uint32_t g = 0, it = 0;
      bool ok = true;
      for (int64_t w = cluster_id; w < n_items && ok; w += n_clusters) {
        int64_t grp; int qb0, len;
        item_range(w, grp, qb0, len);
        for (int k = 0; k < len && ok; ++k, ++it) {
          const uint32_t buf = it & 1, ph = (it >> 1) & 1;
          if (!ptx::mbar_wait(&acc_empty[buf], ph ^ 1)) { atomicExch(p.err_flag, 2); ok = false; break; }
          ptx::tc_fence_after_sync();
          const uint32_t d_tmem = tmem_base + buf * FT_TN;
          for (int c = 0; c < nchunks; ++c, ++g) {
            const uint32_t s = g % FT_STAGES, ph2 = (g / FT_STAGES) & 1;
            if (!ptx::mbar_wait(&full[s], ph2)) { atomicExch(p.err_flag, 3); ok = false; break; }
            ptx::tc_fence_after_sync();
            const uint32_t a_ad = ptx::smem_u32(ring + (size_t)s * FT_STAGE_BYTES);
            const uint32_t b_ad = a_ad + FT_A_BYTES;
#pragma unroll
            for (int ks = 0; ks < FT_KC / 16; ++ks)
              ptx::umma_f16(d_tmem, ptx::umma_desc_sw128(a_ad + ks * 32), ptx::umma_desc_sw128(b_ad + ks * 32), idesc,
                            (c | ks) != 0 ? 1u : 0u);
            if (CS == 1) ptx::umma_commit(&empty[s]);
            else ptx::umma_commit_multicast(&empty[s], CMASK);
          }
          if (ok) ptx::umma_commit(&acc_full[buf]);
        }
      }
    }
  } else {
    // ===== epilogue (warps 2..9; TMEM lane group = warp % 4; warps 2-5 take columns 0..127, warps 6-9 the rest) =====
    const int lg = warp & 3;
    const int chalf = (warp - 2) >> 2;
    const int etid = tid - 64;  // 0..255
    const float inv = p.consts[FC_INV];
    const float sdsq = p.consts[FC_SD] * p.consts[FC_SQ];  // power of two: thresholds move to accumulator units exactly
    uint32_t it = 0;
    bool ok = true;
    for (int64_t w = cluster_id; w < n_items && ok; w += n_clusters) {
      int64_t grp; int qb0, len;
      item_range(w, grp, qb0, len);
      const int64_t tile = p.tile_begin + grp * CS + crank;
      const int64_t doc = tile * FT_TM + lg * 32 + lane;
      const bool doc_ok = doc < p.n_end && tile < p.tile_end;
      for (int k = 0; k < len && ok; ++k, ++it) {
        const int qb = qb0 + (k + stagger) % len;
        const uint32_t buf = it & 1, ph = (it >> 1) & 1;
        // thresholds of this query block (tau is fixed during a chunk; stale values only admit more)
        float* thr = s_thr + buf * FT_TN;
        for (int j = etid; j < FT_TN; j += 32 * FT_EPI_WARPS) {
          const int q = qb * FT_TN + j;
          thr[j] = q < p.nq ? (p.tau[q] - p.margin[q]) * sdsq : CUDART_INF_F;
        }
        asm volatile("bar.sync 1, %0;" ::"n"(32 * FT_EPI_WARPS) : "memory");
        if (!ptx::mbar_wait_backoff(&acc_full[buf], ph, 64)) { atomicExch(p.err_flag, 4); ok = false; break; }
        ptx::tc_fence_after_sync();
        const uint32_t taddr = tmem_base + buf * FT_TN + ((uint32_t)(lg * 32) << 16);
        // Appends of one 32x32 block (32 documents = lanes, 32 queries = columns).  Lane j owns column j: it gets
        // the mask of passing documents, makes ONE atomicAdd for the column (all columns of the block in flight
        // together: one atomic round trip per block, not per column), then the passing lanes store.
        auto store_col = [&](int col, unsigned mk, int j, int base_l, unsigned mym, float acc) {
          const int b0 = __shfl_sync(MEVI_FULL_MASK, base_l, j);
          const unsigned m = __shfl_sync(MEVI_FULL_MASK, mym, j);
          if ((mk >> j) & 1u) {
            const int q = qb * FT_TN + col;
            const int slot = b0 + __popc(m & ((1u << lane) - 1u));
            if (slot < p.capg) {
              p.cand_score[(int64_t)q * p.capg + slot] = acc * inv;
              p.cand_id[(int64_t)q * p.capg + slot] = (int32_t)doc;
            } else {
              *p.overflow = 1;
            }
          }
        };
        // The common case (no document of this warp beats any of the 32 thresholds) must cost ~1 instruction per
        // accumulator: vector threshold loads, one predicate per element, ONE vote per 32 columns.  The next 32
        // columns are already on their way from tensor memory while these are tested.
        auto test32 = [&](const uint32_t (&r)[32], int c0) {
          const float4* t4 = reinterpret_cast<const float4*>(thr + c0);
          bool any = false;
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4) {
            const float4 t = t4[j4];
            any |= !(__uint_as_float(r[4 * j4 + 0]) < t.x);
            any |= !(__uint_as_float(r[4 * j4 + 1]) < t.y);
            any |= !(__uint_as_float(r[4 * j4 + 2]) < t.z);
            any |= !(__uint_as_float(r[4 * j4 + 3]) < t.w);
          }
          if (!__any_sync(MEVI_FULL_MASK, any && doc_ok)) return;
          // some document passes: per-lane column mask, then only the columns that have a passing document
          unsigned mk = 0;
#pragma unroll
          for (int j = 0; j < 32; ++j) mk |= (!(__uint_as_float(r[j]) < thr[c0 + j]) ? 1u : 0u) << j;
          if (!doc_ok) mk = 0;
          const unsigned cols = __reduce_or_sync(MEVI_FULL_MASK, mk);
          const bool dense = __popc(cols) > 10;  // first chunks: most columns pass somewhere
          unsigned mym = 0;  // lane j: documents (lanes) passing column j
          if (dense) {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const unsigned m = __ballot_sync(MEVI_FULL_MASK, (mk >> j) & 1u);
              if (lane == j) mym = m;
            }
          } else {
            for (unsigned c = cols; c; c &= c - 1) {  // warp-uniform
              const int j = __ffs(c) - 1;
              const unsigned m = __ballot_sync(MEVI_FULL_MASK, (mk >> j) & 1u);
              if (lane == j) mym = m;
            }
          }
          int base_l = 0;
          if (mym) base_l = atomicAdd(&p.count[qb * FT_TN + c0 + lane], __popc(mym));
          if (dense) {
#pragma unroll
            for (int j = 0; j < 32; ++j) store_col(c0 + j, mk, j, base_l, mym, __uint_as_float(r[j]));
          } else {
            for (unsigned c = cols; c; c &= c - 1) {
              const int j = __ffs(c) - 1;
              // r[j] for a run-time j without spilling r[] to local memory: 5-level select tree
              uint32_t a16[16], a8[8], a4[4], a2[2];
#pragma unroll
              for (int i = 0; i < 16; ++i) a16[i] = (j & 16) ? r[i + 16] : r[i];
#pragma unroll
              for (int i = 0; i < 8; ++i) a8[i] = (j & 8) ? a16[i + 8] : a16[i];
#pragma unroll
              for (int i = 0; i < 4; ++i) a4[i] = (j & 4) ? a8[i + 4] : a8[i];
#pragma unroll
              for (int i = 0; i < 2; ++i) a2[i] = (j & 2) ? a4[i + 2] : a4[i];
              const uint32_t v = (j & 1) ? a2[1] : a2[0];
              store_col(c0 + j, mk, j, base_l, mym, __uint_as_float(v));
            }
          }
        };
        uint32_t ra[32], rb[32];
        const int cbeg = chalf * (FT_TN / 2), cend = cbeg + FT_TN / 2;
        ptx::tmem_ld32(taddr + cbeg, ra);
#pragma unroll 1
        for (int c0 = cbeg; c0 < cend; c0 += 64) {
          ptx::tmem_ld_wait();
          ptx::tmem_ld32(taddr + c0 + 32, rb);
          test32(ra, c0);
          ptx::tmem_ld_wait();
          if (c0 + 64 < cend) ptx::tmem_ld32(taddr + c0 + 64, ra);
          test32(rb, c0 + 32);
        }
        ptx::tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&acc_empty[buf]);
      }
    }
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  if (CS > 1) ptx::cluster_sync_all();  // no CTA leaves while peers may still multicast into it
  if (warp == 0) ptx::tmem_dealloc(tmem_base, 512);
}

template <int CS>
int launch_flat_gemm(mevi_ctx* ctx, const GemmParams& p, size_t smem, int max_clusters, cudaStream_t st) {
  MEVI_CUDA(ctx, cudaFuncSetAttribute(flat_gemm_kernel<CS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t groups = (p.tile_end - p.tile_begin + CS - 1) / CS;
  const int64_t items = groups * p.qparts;
  const int clusters = (int)(items < max_clusters ? items : max_clusters);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(clusters * CS));
  cfg.blockDim = dim3(FT_THREADS2);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CS;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  MEVI_CUDA(ctx, cudaLaunchKernelEx(&cfg, flat_gemm_kernel<CS>, p));
  return MEVI_OK;
}

// co-resident clusters of CS CTAs (1 CTA per SM): 148/CS unless a GPC cannot be tiled exactly
template <int CS>
int flat_max_clusters(mevi_ctx* ctx, size_t smem) {
  if (CS == 1) return ctx->sm_count;
  if (cudaFuncSetAttribute(flat_gemm_kernel<CS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return 0;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(ctx->sm_count / CS * CS));
  cfg.blockDim = dim3(FT_THREADS2);
  cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CS;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, flat_gemm_kernel<CS>, &cfg) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

// one CTA per query: tau = k-th best approximate score of (kept + newly appended) candidates, found by a radix SELECT
// over the bits in which the scores differ (block256_select_kth, common.cuh; no sort: the list is consumed as a set); everything inside the margin window
// [tau - margin, inf) is kept, the rest can never reach the exact top-k (tau only rises) and is dropped.  More than
// `keep` candidates inside the window breaks the guarantee -> overflow flag
// (`ov_stride` = 0: one flag for the call - flat search; 1: a flag per query - grouped re-rank, which re-runs only the
// affected queries through the streaming kernel).  The kept list is NOT ordered.
__global__ void __launch_bounds__(256) flat_tensor_compact_kernel(float* tau, const float* margin, int* count, float* cand_score,
                                                                  int32_t* cand_id, int* overflow, int capg, int k, int keep,
                                                                  int ov_stride) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* s_score = reinterpret_cast<float*>(smem_raw);                 // [capg]
  float* s_ks = s_score + capg;                                        // [keep]
  int32_t* s_ki = reinterpret_cast<int32_t*>(s_ks + keep);             // [keep]
  unsigned* s_hist = reinterpret_cast<unsigned*>(s_ki + keep);         // [256]
  __shared__ unsigned s_scratch[4];
  __shared__ int s_n;
  const int q = blockIdx.x, tid = threadIdx.x;
  int cnt = count[q];
  if (cnt > capg) cnt = capg;
  if (cnt == 0) return;
  if (tid == 0) s_n = 0;
  for (int i = tid; i < cnt; i += blockDim.x) s_score[i] = cand_score[(int64_t)q * capg + i];
  __syncthreads();
  float t = tau[q];
  // never below a bound the caller already had (the grouped re-rank starts from a lower bound of the k-th score)
  if (cnt >= k) t = fmaxf(t, block256_select_kth(s_score, cnt, k, s_hist, s_scratch));
  const float window = t - margin[q];
  for (int i = tid; i < cnt; i += blockDim.x) {
    const float sc = s_score[i];
    if (!(sc < window)) {
      const int pos = atomicAdd(&s_n, 1);
      if (pos < keep) { s_ks[pos] = sc; s_ki[pos] = cand_id[(int64_t)q * capg + i]; }
    }
  }
  __syncthreads();
  const int n_in = s_n;
  const int kept = n_in < keep ? n_in : keep;
  for (int i = tid; i < kept; i += blockDim.x) {
    cand_score[(int64_t)q * capg + i] = s_ks[i];
    cand_id[(int64_t)q * capg + i] = s_ki[i];
  }
  if (tid == 0) {
    count[q] = kept;
    tau[q] = t;
    if (n_in > keep) overflow[(int64_t)q * ov_stride] = 1;
  }
}

// one CTA per query: exact fp32 re-score of the surviving candidates, sort, emit the k best
__global__ void __launch_bounds__(256) flat_rescore_kernel(const float* __restrict__ Q, const float* __restrict__ D, int d,
                                                           const int* __restrict__ count, const int32_t* __restrict__ cand_id,
                                                           const float* __restrict__ cand_score, const float* __restrict__ tau,
                                                           const float* __restrict__ margin,
                                                           int capg, int k, int keep_pow2, int64_t id_base,
                                                           float* __restrict__ scores, int64_t* __restrict__ ids) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* s_score = reinterpret_cast<float*>(smem_raw);
  int32_t* s_id = reinterpret_cast<int32_t*>(s_score + keep_pow2);
  const int q = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int cnt = count[q];
  if (cnt > keep_pow2) cnt = keep_pow2;
  for (int i = threadIdx.x; i < keep_pow2; i += blockDim.x) {
    s_score[i] = -CUDART_INF_F;
    s_id[i] = 0x7fffffff;
  }
  __syncthreads();
  // a member of the exact top-k has an approximate score >= (k-th approximate score) - margin: the rest of the kept
  // list (unordered; kept under an earlier, lower threshold) cannot matter and is not fetched
  const float window = tau[q] - margin[q];
  for (int i = warp; i < cnt; i += 8) {
    if (cand_score[(int64_t)q * capg + i] < window) continue;
    const int32_t row = cand_id[(int64_t)q * capg + i];
    float acc = 0.f;
    for (int c4 = lane * 4; c4 < d; c4 += 128) {  // same summation pattern as the dense scorer
      const float4 a = ldg_f4(Q + (int64_t)q * d + c4);
      const float4 b = ld_stream_f4(D + (int64_t)row * d + c4);
      acc = fmaf(a.x, b.x, acc);
      acc = fmaf(a.y, b.y, acc);
      acc = fmaf(a.z, b.z, acc);
      acc = fmaf(a.w, b.w, acc);
    }
    acc = warp_sum(acc);
    if (lane == 0) {
      s_score[i] = acc;
      s_id[i] = row;
    }
  }
  __syncthreads();
  block_bitonic_sort<int32_t>(s_score, s_id, keep_pow2);
  for (int i = threadIdx.x; i < k; i += blockDim.x) {
    // kept candidates below the window were not re-scored (thresholds can rise after the last compaction when ranks
    // share them): they sorted behind every scored one and are not results
    const bool ok = i < cnt && s_id[i] != 0x7fffffff;
    scores[(int64_t)q * k + i] = ok ? s_score[i] : -CUDART_INF_F;
    ids[(int64_t)q * k + i] = ok ? id_base + (int64_t)s_id[i] : -1;
  }
}

__global__ void flat_tensor_init_kernel(float* tau, int* count, int* overflow, int* err, int nq) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nq) {
    tau[i] = -CUDART_INF_F;
    count[i] = 0;
  }
  if (i == 0) {
    *overflow = 0;
    *err = 0;
  }
}

}  // namespace

bool mevi_flat_tensor_supported(mevi_ctx* ctx, int d, int k) {
  // k <= 256: 512 approximate candidates kept per query in 4,096-slot buffers; k <= 1,024 (the reference CLI default is
  // --topk 1000, faiss_search.py:88): 2,048 kept in 8,192-slot buffers
  return ctx && ctx->cc_major == 10 && d >= FT_KC && d % FT_KC == 0 && d <= 4096 && k >= 1 && k <= 1024;
}

namespace {
// fp16 image of a document matrix + its metadata (the "add" half of a flat index)
int flat_docs_prepare(mevi_ctx* ctx, const float* D, int64_t n, int d, __half* Aimg, unsigned* docmeta, cudaStream_t st) {
  const int64_t n_tiles = (n + FT_TM - 1) / FT_TM;
  MEVI_CUDA(ctx, cudaMemsetAsync(docmeta, 0, DM_NUM * sizeof(unsigned), st));
  const int64_t sample_rows = 4096;
  flat_absmax_kernel<<<ctx->sm_count, 256, 0, st>>>(D, n, d, n > sample_rows ? n / sample_rows : 1, docmeta + DM_ABSMAX);
  flat_doc_scale_kernel<<<1, 32, 0, st>>>(docmeta);
  to_fp16_image_kernel<<<ctx->sm_count * 8, 256, 0, st>>>(D, n, d, FT_TM, reinterpret_cast<const float*>(docmeta), DM_SCALE, Aimg, nullptr,
                                                          docmeta + DM_MAXNORM, reinterpret_cast<int*>(docmeta + DM_CLAMPED),
                                                          n_tiles * FT_TM);
  MEVI_CUDA(ctx, cudaGetLastError());
  MEVI_COUNT_LAUNCH(ctx, 3);
  return MEVI_OK;
}
}  // namespace

int mevi_flat_tensor_search_image(mevi_ctx* ctx, const float* Q, int nq, const float* D, int64_t n, int d, const __half* Aimg,
                                  const unsigned* docmeta, int k, int64_t id_base, float* scores, int64_t* ids, int* fell_back,
                                  cudaStream_t st);

// Returns MEVI_OK with *fell_back = 0 when scores/ids hold the exact answer; *fell_back = 1 when the
// guarantee could not be established (margin overflow, fp16 clamp, pipeline time-out): the caller then
// runs the fp32 search.
int mevi_flat_tensor_search(mevi_ctx* ctx, const float* Q, int nq, const float* D, int64_t n, int d, int k,
                            int64_t id_base, float* scores, int64_t* ids, int* fell_back, cudaStream_t st) {
  // one-shot form: the image lives in scratch memory and is rebuilt by every call (a caller that searches the same
  // documents again holds a mevi_flat_index instead)
  *fell_back = 1;
  const int64_t n_tiles = (n + FT_TM - 1) / FT_TM;
  const size_t img_bytes = (size_t)n_tiles * FT_TM * d * 2;
  char* ws = (char*)mevi_ws(ctx, WS_FLAT_IMAGE, img_bytes + 256);
  if (!ws) return MEVI_ERR_NOMEM;
  unsigned* docmeta = (unsigned*)ws;
  __half* Aimg = (__half*)(ws + 256);
  int rc = flat_docs_prepare(ctx, D, n, d, Aimg, docmeta, st);
  if (rc != MEVI_OK) return rc;
  return mevi_flat_tensor_search_image(ctx, Q, nq, D, n, d, Aimg, docmeta, k, id_base, scores, ids, fell_back, st);
}

int mevi_flat_tensor_search_image(mevi_ctx* ctx, const float* Q, int nq, const float* D, int64_t n, int d, const __half* Aimg,
                                  const unsigned* docmeta, int k, int64_t id_base, float* scores, int64_t* ids, int* fell_back,
                                  cudaStream_t st) {
  *fell_back = 1;
  const int nchunks = d / FT_KC;
  const int64_t n_tiles = (n + FT_TM - 1) / FT_TM;
  const int n_qblocks = (nq + FT_TN - 1) / FT_TN;
  const int keep = k <= FT_KEEP / 2 ? FT_KEEP : 2048;
  const int capg = k <= FT_KEEP / 2 ? 4096 : 8192;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = (off + bytes + 255) & ~size_t(255); return o; };
  const size_t o_consts = take(FC_NUM * 4), o_abs = take(16), o_flags = take(16), o_tau = take((size_t)nq * 4),
               o_margin = take((size_t)nq * 4), o_qnorm = take((size_t)nq * 4), o_cnt = take((size_t)nq * 4),
               o_cs = take((size_t)nq * capg * 4), o_ci = take((size_t)nq * capg * 4),
               o_bimg = take((size_t)n_qblocks * FT_TN * d * 2);
  char* ws = (char*)mevi_ws(ctx, WS_TOPK_PART, off);
  if (!ws) return MEVI_ERR_NOMEM;
  float* consts = (float*)(ws + o_consts);
  unsigned* absmax_q = (unsigned*)(ws + o_abs);       // Q absmax
  int* flags = (int*)(ws + o_flags);                   // [0] overflow, [1] pipeline error, [2] a Q element clamped
  float* tau = (float*)(ws + o_tau);
  float* margin = (float*)(ws + o_margin);
  float* qnorm = (float*)(ws + o_qnorm);
  int* count = (int*)(ws + o_cnt);
  float* cand_score = (float*)(ws + o_cs);
  int32_t* cand_id = (int32_t*)(ws + o_ci);
  __half* Bimg = (__half*)(ws + o_bimg);

  MEVI_CUDA(ctx, cudaMemsetAsync(ws + o_abs, 0, 32 + 256, st));  // absmax_q + flags
  flat_tensor_init_kernel<<<(nq + 255) / 256, 256, 0, st>>>(tau, count, flags, flags + 1, nq);
  flat_absmax_kernel<<<ctx->sm_count, 256, 0, st>>>(Q, nq, d, 1, absmax_q);
  flat_consts_kernel<<<1, 32, 0, st>>>(docmeta, absmax_q, consts);
  to_fp16_image_kernel<<<ctx->sm_count * 2, 256, 0, st>>>(Q, nq, d, FT_TN, consts, FC_SQ, Bimg, qnorm, nullptr, flags + 2,
                                                          (int64_t)n_qblocks * FT_TN);
  flat_margin_kernel<<<(nq + 255) / 256, 256, 0, st>>>(qnorm, nq, d, docmeta + DM_MAXNORM, consts, margin);
  MEVI_CUDA(ctx, cudaGetLastError());
  MEVI_COUNT_LAUNCH(ctx, 5);

  GemmParams p;
  p.Aimg = Aimg; p.Bimg = Bimg; p.nq = nq; p.n_qblocks = n_qblocks; p.nchunks = nchunks; p.n_end = n;
  p.consts = consts; p.tau = tau; p.margin = margin; p.count = count; p.cand_score = cand_score; p.cand_id = cand_id;
  p.overflow = flags; p.capg = capg; p.err_flag = flags + 1;
  const size_t smem_gemm = (size_t)FT_STAGES * FT_STAGE_BYTES + 2 * FT_TN * 4 + (2 * FT_STAGES + 4) * 8 + 16 + 1024;
  // cluster size: FT_DEFAULT_CLUSTER, or 1 when no cluster of that size can be resident
  int cs = FT_DEFAULT_CLUSTER;
  int max_clusters = cs == 4 ? flat_max_clusters<4>(ctx, smem_gemm) : cs == 2 ? flat_max_clusters<2>(ctx, smem_gemm) : 0;
  if (max_clusters <= 0) { cs = 1; max_clusters = ctx->sm_count; }
  const size_t smem_compact = (size_t)capg * 8;
  MEVI_CUDA(ctx, cudaFuncSetAttribute(flat_tensor_compact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_compact));

  // chunks of document tiles growing geometrically: the first (no thresholds yet, every score is appended) is small,
  // so its compaction sorts 1,024 (2,048 for k > 256) and not `capg` candidates per query; it can never overflow the
  // candidate buffers
  int64_t chunk_tiles = k <= FT_KEEP / 2 ? 8 : 16;
  static_assert(8 * FT_TM <= 4096 - FT_KEEP && 16 * FT_TM <= 8192 - 2048, "first chunk must fit the candidate buffer");
  int64_t pos = 0;
  while (pos < n_tiles) {
    const int64_t end = pos + chunk_tiles < n_tiles ? pos + chunk_tiles : n_tiles;
    p.tile_begin = pos;
    p.tile_end = end;
    {  // enough work items for ~3 per cluster: split the query-block range of a tile group when groups are few
      const int64_t groups = (end - pos + cs - 1) / cs;
      int64_t parts = groups >= 3 * (int64_t)max_clusters ? 1 : (3 * (int64_t)max_clusters + groups - 1) / groups;
      p.qparts = (int)(parts > n_qblocks ? n_qblocks : parts);
    }
    const int rc = cs == 4 ? launch_flat_gemm<4>(ctx, p, smem_gemm, max_clusters, st)
                 : cs == 2 ? launch_flat_gemm<2>(ctx, p, smem_gemm, max_clusters, st)
                           : launch_flat_gemm<1>(ctx, p, smem_gemm, max_clusters, st);
    if (rc != MEVI_OK) return rc;
    flat_tensor_compact_kernel<<<nq, 256, smem_compact, st>>>(tau, margin, count, cand_score, cand_id, flags, capg, k, keep, 0);
    MEVI_CUDA(ctx, cudaGetLastError());
    MEVI_COUNT_LAUNCH(ctx, 2);
    pos = end;
    int64_t next = pos * 3;
    const int64_t cap_chunk = ((int64_t)1 << 22) / FT_TM;
    chunk_tiles = next > cap_chunk ? cap_chunk : next;
  }
  int h_flags[4] = {0, 0, 0, 0};
  unsigned h_docmeta[DM_NUM] = {0, 0, 0, 0};
  MEVI_CUDA(ctx, cudaMemcpyAsync(h_flags, flags, sizeof(h_flags), cudaMemcpyDeviceToHost, st));
  MEVI_CUDA(ctx, cudaMemcpyAsync(h_docmeta, docmeta, sizeof(h_docmeta), cudaMemcpyDeviceToHost, st));
  MEVI_CUDA(ctx, cudaStreamSynchronize(st));
  if (int drc = mevi_deferred_error(ctx)) return drc;  // a kernel of this (or an earlier asynchronous) launch timed out
  if (h_flags[1]) return mevi_set_error(ctx, MEVI_ERR_CUDA, "flat tensor kernel pipeline time-out (code %d)", h_flags[1]);
  if (h_flags[0] || h_flags[2] || h_docmeta[DM_CLAMPED]) return MEVI_OK;  // guarantee not established: caller falls back to fp32
  const size_t smem_rescore = (size_t)keep * 8;
  MEVI_CUDA(ctx, cudaFuncSetAttribute(flat_rescore_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_rescore));
  flat_rescore_kernel<<<nq, 256, smem_rescore, st>>>(Q, D, d, count, cand_id, cand_score, tau, margin, capg, k, keep, id_base, scores,
                                                     ids);
  MEVI_CUDA(ctx, cudaGetLastError());
  MEVI_COUNT_LAUNCH(ctx, 1);
  *fell_back = 0;
  return MEVI_OK;
}

// =====================================================================================================
// K3g — cluster-restricted re-rank as LEAF-GROUPED GEMMs on the tensor cores.
//
// The streaming kernel of rerank.cu reads every candidate row once per query that selected its leaf
// (main_models.py:3915-4014 does the same, one matmul per (query, leaf)).  With L = 100 leaves a query
// scores ~150k documents, and a leaf is selected by ~30 queries, so the rows of a leaf can be read ONCE
// and scored against all the queries that selected it: per leaf a [docs of the leaf] x [queries that
// chose it] GEMM.  Same numerics contract as K2: fp16 tcgen05 scores are a prefilter with a rigorous
// margin, survivors are re-scored in exact fp32 in the dense scorer's summation order, and anything
// that cannot be guaranteed (margin window overflow, fp16 clamp) makes the caller fall back to the
// streaming kernel.
//   index side (once): document tiles of 128 rows that never straddle a leaf (tile_row0 / tile_nrows),
//     fp16 image [tile][K chunk][128][64] of the leaf-ordered matrix;
//   call side: (leaf, query) pairs sorted by leaf and cut into groups of <= 64 queries (group_qid),
//     work items (tile of the leaf, group of the leaf); thresholds start from a lower bound tau0 of every
//     query's k-th best score (exact top-k of a prefix of its candidates, mevi_cluster_rerank_prefix) and
//     tighten between rounds of pairs, exactly like the chunks of the flat search.
// GEMM CTA: 320 threads, A 16 KB + B 8 KB per stage, 8 stages, tcgen05.mma M=128 N=64 K=16, two 64-column
// accumulator buffers in TMEM, 8 epilogue warps (lane group x 32-column half).
namespace {

constexpr int GR_TN = 64;   // columns (queries) per group
constexpr int GR_B_BYTES = GR_TN * 128;
constexpr int GR_EPI_WARPS = 8;
constexpr int GR_THREADS = 64 + 32 * GR_EPI_WARPS;
constexpr int GR_CAPG = 8192;  // candidate slots per query between compactions (512 kept + what a round appends)
// A work item = one document tile x up to MAXG CONSECUTIVE column groups of its leaf (item_group packs the first group in
// its low 24 bits and the number of groups in the bits above; 0 = 1).  The tile's 196 KB then come through L2 once for
// MAXG * 64 queries.  The ring is cut for the widest item of the instantiation: MAXG 1 -> 8 stages x 24 KB (the sample
// rounds, whose items are one thin group), 2 -> 6 x 32 KB, 4 -> 4 x 48 KB (the last round: every tile of a leaf against
// all the queries that chose it).
constexpr int gr_stage_bytes(int maxg) { return FT_A_BYTES + maxg * GR_B_BYTES; }
constexpr int gr_stages(int maxg) { return maxg == 1 ? 8 : (maxg == 2 ? 6 : 4); }
constexpr uint32_t GR_GROUP_MASK = 0xFFFFFFu;

struct GroupedParams {
  const __half* Aimg; const __half* Bimg;
  const int32_t* item_tile; const int32_t* item_group; int64_t n_items;
  const int32_t* tile_row0; const int32_t* tile_nrows;
  const int32_t* group_qid;  // [n_groups][GR_TN], -1 = padding
  const int32_t* group_ncols; // [n_groups] columns in use, rounded up to 16: a thin group is a narrower GEMM (N = 16 .. 64)
  int nchunks;
  const float* consts; const float* tau; const float* margin;
  int* count; float* cand_score; int32_t* cand_id; int* overflow; int capg;
  int* err_flag;
  // multi-cluster index (MC instantiation only; see "Multi-cluster indexes" below)
  const int32_t* occ; int occ_w;  // [rows][occ_w] CSR leaves of the document's other positions (occurrence table), occ_w = C - 1
  const int32_t* tile_leaf;       // [n_tiles] leaf of every image tile
  const uint64_t* qtab; int qtab_log2;  // [nq][1 << qtab_log2] per-query leaf tables (mc_probe)
  const float* mc_cheap;          // [nq] factor applied to a positive threshold for the one-compare prefilter
  int aggr;                       // MEVI_MULTICLUS_ADD / _MAX
};

// ---- Multi-cluster indexes (--doc_multiclus > 1) ----------------------------------------------------------------------
// A document listed under several leaves has several rows of the leaf-ordered matrix (CSR positions).  For a query q
// and a document, c = the number of positions of q's leaf list whose leaf lists the document; the kept occurrence is
// the canonical one of rerank.cu: the earliest position of the list, the first CSR position inside that leaf.  Per query
// an open-addressed table (1 << qtab_log2 >= 2L slots, rerank.cu's hash) maps a leaf to one 64-bit word: leaf (bits
// 0-31; 0xFFFFFFFF = empty), its first position in the list (32-47) and its number of positions (48-63).
__device__ __forceinline__ uint64_t mc_probe(const uint64_t* __restrict__ tab, int log2, int leaf) {
  const unsigned mask = (1u << log2) - 1u;
  unsigned h = ((unsigned)leaf * 0x9E3779B1u) >> (32 - log2);
  for (;;) {  // load factor <= 1/2: an empty slot ends every probe sequence
    const uint64_t e = __ldg(tab + h);
    if ((uint32_t)e == (uint32_t)leaf || (uint32_t)e == 0xFFFFFFFFu) return e;
    h = (h + 1) & mask;
  }
}

// c of the occurrence (row of leaf `own`, query with table `tab`), or -1 when the occurrence is not canonical.  `own`
// sits at its first position in the list (the plan holds one pair per distinct leaf).
__device__ __forceinline__ int mc_count(const uint64_t* __restrict__ tab, int log2, int own, const int32_t* __restrict__ sib,
                                        int w) {
  const uint64_t e = mc_probe(tab, log2, own);
  const int t = (int)((e >> 32) & 0xFFFFu);
  int c = (int)(e >> 48);
  for (int i = 0; i < w; ++i) {
    const int32_t leaf = __ldg(sib + i);
    if (leaf == -1) break;              // padding
    if (leaf <= -2) return -1;          // an earlier CSR position of the same leaf
    const uint64_t f = mc_probe(tab, log2, leaf);
    if ((uint32_t)f == 0xFFFFFFFFu) continue;  // a leaf the query did not ask for
    if ((int)((f >> 32) & 0xFFFFu) < t) return -1;
    c += (int)(f >> 48);
  }
  return c;
}

// the reference's 'add': zeros, then += s once per position (main_models.py:4004-4007), as in rerank.cu
__device__ __forceinline__ float mc_fold(float s, int c) {
  float a = 0.f;
  for (int i = 0; i < c; ++i) a = __fadd_rn(a, s);
  return a;
}

template <int MAXG, bool MC>
__global__ void __launch_bounds__(GR_THREADS, 1) grouped_gemm_kernel(GroupedParams p) {
  constexpr int STAGES = gr_stages(MAXG), STAGE_BYTES = gr_stage_bytes(MAXG), ACC_COLS = MAXG * GR_TN;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* ring = smem;  // [STAGES][A 16 KB | B MAXG x 8 KB]
  float* s_thr = reinterpret_cast<float*>(smem + (size_t)STAGES * STAGE_BYTES);  // [2][ACC_COLS]
  int* s_qid = reinterpret_cast<int*>(s_thr + 2 * ACC_COLS);                      // [2][ACC_COLS]
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_qid + 2 * ACC_COLS);
  uint64_t* full = bars;
  uint64_t* empty = full + STAGES;
  uint64_t* acc_full = empty + STAGES;
  uint64_t* acc_empty = acc_full + 2;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(acc_empty + 2);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) { ptx::mbar_init(&full[s], 1); ptx::mbar_init(&empty[s], 1); }
    for (int b = 0; b < 2; ++b) { ptx::mbar_init(&acc_full[b], 1); ptx::mbar_init(&acc_empty[b], GR_EPI_WARPS); }
    ptx::mbar_fence_init();
  }
  if (warp == 0) ptx::tmem_alloc(tmem_holder, 2 * ACC_COLS);
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_holder;
  const int nchunks = p.nchunks;

  if (warp == 0) {
    if (lane == 0) {
      uint32_t g = 0;
      bool ok = true;
      for (int64_t w = blockIdx.x; w < p.n_items && ok; w += gridDim.x) {
        const uint32_t ig = (uint32_t)p.item_group[w];
        const int ng = MAXG == 1 ? 1 : min(max((int)(ig >> 24), 1), MAXG);
        const int64_t grp = ig & GR_GROUP_MASK;
        const uint32_t last_bytes = (uint32_t)p.group_ncols[grp + ng - 1] * 128u;  // rows in use of the last group
        const __half* a_src = p.Aimg + (size_t)p.item_tile[w] * nchunks * FT_TM * FT_KC;
        const __half* b_src = p.Bimg + (size_t)grp * nchunks * GR_TN * FT_KC;
        for (int c = 0; c < nchunks; ++c, ++g) {
          const uint32_t s = g % STAGES, ph = (g / STAGES) & 1;
          if (!ptx::mbar_wait_backoff(&empty[s], ph ^ 1, 32)) { atomicExch(p.err_flag, 1); ok = false; break; }
          ptx::mbar_arrive_expect_tx(&full[s], FT_A_BYTES + (ng - 1) * GR_B_BYTES + last_bytes);
          uint8_t* st_a = ring + (size_t)s * STAGE_BYTES;
          ptx::bulk_g2s(st_a, a_src + (size_t)c * FT_TM * FT_KC, FT_A_BYTES, &full[s]);
#pragma unroll
          for (int j = 0; j < MAXG; ++j)
            if (j < ng)
              ptx::bulk_g2s(st_a + FT_A_BYTES + j * GR_B_BYTES, b_src + ((size_t)j * nchunks + c) * GR_TN * FT_KC,
                            j == ng - 1 ? last_bytes : (uint32_t)GR_B_BYTES, &full[s]);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      uint32_t g = 0, it = 0;
      bool ok = true;
      for (int64_t w = blockIdx.x; w < p.n_items && ok; w += gridDim.x, ++it) {
        const uint32_t ig = (uint32_t)p.item_group[w];
        const int ng = MAXG == 1 ? 1 : min(max((int)(ig >> 24), 1), MAXG);
        const uint32_t idesc = ptx::umma_idesc_f16_m128(GR_TN * (ng - 1) + p.group_ncols[(ig & GR_GROUP_MASK) + ng - 1]);
        const uint32_t buf = it & 1, ph = (it >> 1) & 1;
        if (!ptx::mbar_wait(&acc_empty[buf], ph ^ 1)) { atomicExch(p.err_flag, 2); ok = false; break; }
        ptx::tc_fence_after_sync();
        const uint32_t d_tmem = tmem_base + buf * ACC_COLS;
        for (int c = 0; c < nchunks; ++c, ++g) {
          const uint32_t s = g % STAGES, ph2 = (g / STAGES) & 1;
          if (!ptx::mbar_wait(&full[s], ph2)) { atomicExch(p.err_flag, 3); ok = false; break; }
          ptx::tc_fence_after_sync();
          const uint32_t a_ad = ptx::smem_u32(ring + (size_t)s * STAGE_BYTES);
          const uint32_t b_ad = a_ad + FT_A_BYTES;
#pragma unroll
          for (int ks = 0; ks < FT_KC / 16; ++ks)
            ptx::umma_f16(d_tmem, ptx::umma_desc_sw128(a_ad + ks * 32), ptx::umma_desc_sw128(b_ad + ks * 32), idesc,
                          (c | ks) != 0 ? 1u : 0u);
          ptx::umma_commit(&empty[s]);
        }
        if (ok) ptx::umma_commit(&acc_full[buf]);
      }
    }
  } else {
    // ===== epilogue: warp -> (TMEM lane group = warp % 4, 32-column half of every 64-column group) =====
    const int lg = warp & 3;
    const int ch = ((warp - 2) >> 2) * 32;
    const int etid = tid - 64;
    const float inv = p.consts[FC_INV];
    const float sdsq = p.consts[FC_SD] * p.consts[FC_SQ];
    uint32_t it = 0;
    bool ok = true;
    for (int64_t w = blockIdx.x; w < p.n_items && ok; w += gridDim.x, ++it) {
      const int tile = p.item_tile[w];
      const uint32_t ig = (uint32_t)p.item_group[w];
      const int ng = MAXG == 1 ? 1 : min(max((int)(ig >> 24), 1), MAXG);
      const int64_t grp = ig & GR_GROUP_MASK;
      const uint32_t buf = it & 1, ph = (it >> 1) & 1;
      float* thr = s_thr + buf * ACC_COLS;
      int* qid = s_qid + buf * ACC_COLS;
      if (etid < GR_TN * ng) {
        const int q = p.group_qid[grp * GR_TN + etid];
        qid[etid] = q;
        float t = q >= 0 ? (p.tau[q] - p.margin[q]) * sdsq : CUDART_INF_F;
        // MC 'add': an aggregated score is at most max(s, c_max s) (rounded up), so a positive threshold is divided
        // by c_max (mc_cheap < 1 / c_max) and ONE compare per accumulator still decides who goes further
        if constexpr (MC) if (q >= 0 && t > 0.f) t *= p.mc_cheap[q];
        thr[etid] = t;
      }
      asm volatile("bar.sync 1, %0;" ::"n"(32 * GR_EPI_WARPS) : "memory");
      if (!ptx::mbar_wait_backoff(&acc_full[buf], ph, 64)) { atomicExch(p.err_flag, 4); ok = false; break; }
      ptx::tc_fence_after_sync();
      const int r = lg * 32 + lane;
      const bool doc_ok = r < p.tile_nrows[tile];
      const int32_t doc = p.tile_row0[tile] + r;  // row of the leaf-ordered matrix
      const int nlast = p.group_ncols[grp + ng - 1];
      for (int sg = 0; sg < ng; ++sg) {
        const int c0 = sg * GR_TN + ch;
        const bool in_use = sg < ng - 1 || ch < nlast;  // this warp's 32 columns of a thin last group may not exist
        uint32_t acc[32];
        if (in_use) {
          ptx::tmem_ld32(tmem_base + buf * ACC_COLS + c0 + ((uint32_t)(lg * 32) << 16), acc);
          ptx::tmem_ld_wait();
        }
        if (sg == ng - 1) {  // the last accumulators are in registers: hand the buffer back first
          ptx::tc_fence_before_sync();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&acc_empty[buf]);
        }
        if (!in_use) continue;
        const float4* t4 = reinterpret_cast<const float4*>(thr + c0);
        bool any = false;
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) {
          const float4 t = t4[j4];
          any |= !(__uint_as_float(acc[4 * j4 + 0]) < t.x);
          any |= !(__uint_as_float(acc[4 * j4 + 1]) < t.y);
          any |= !(__uint_as_float(acc[4 * j4 + 2]) < t.z);
          any |= !(__uint_as_float(acc[4 * j4 + 3]) < t.w);
        }
        if (__any_sync(MEVI_FULL_MASK, any && doc_ok)) {
          unsigned mk = 0;
#pragma unroll
          for (int j = 0; j < 32; ++j) mk |= (!(__uint_as_float(acc[j]) < thr[c0 + j]) ? 1u : 0u) << j;
          if (!doc_ok) mk = 0;
          if constexpr (MC) {
            // the few pairs that passed: drop non-canonical occurrences, aggregate over the query's WHOLE leaf list, apply
            // the exact test to the aggregated approximate score and append that score.  One column at a time.
            const int own = p.tile_leaf[tile];
            const int32_t* sib = p.occ + (int64_t)doc * p.occ_w;
            const unsigned tab_sz = 1u << p.qtab_log2;
            for (unsigned cols = __reduce_or_sync(MEVI_FULL_MASK, mk); cols; cols &= cols - 1) {  // warp-uniform
              const int j = __ffs(cols) - 1;
              const int q = qid[c0 + j];
              bool pass = ((mk >> j) & 1u) && q >= 0;
              float agg = 0.f;
              if (pass) {
                // acc[j] for a run-time j without spilling acc[] to local memory: 5-level select tree
                uint32_t a16[16], a8[8], a4[4], a2[2];
#pragma unroll
                for (int i = 0; i < 16; ++i) a16[i] = (j & 16) ? acc[i + 16] : acc[i];
#pragma unroll
                for (int i = 0; i < 8; ++i) a8[i] = (j & 8) ? a16[i + 8] : a16[i];
#pragma unroll
                for (int i = 0; i < 4; ++i) a4[i] = (j & 4) ? a8[i + 4] : a8[i];
#pragma unroll
                for (int i = 0; i < 2; ++i) a2[i] = (j & 2) ? a4[i + 2] : a4[i];
                const float s = __uint_as_float((j & 1) ? a2[1] : a2[0]) * inv;
                const int c = mc_count(p.qtab + (int64_t)q * tab_sz, p.qtab_log2, own, sib, p.occ_w);
                agg = p.aggr == MEVI_MULTICLUS_ADD ? mc_fold(s, c) : s;
                pass = c >= 0 && !(agg < p.tau[q] - p.margin[q]);
              }
              const unsigned m = __ballot_sync(MEVI_FULL_MASK, pass);
              if (m) {
                int b0 = 0;
                if (lane == 0) b0 = atomicAdd(&p.count[q], __popc(m));
                b0 = __shfl_sync(MEVI_FULL_MASK, b0, 0);
                if (pass) {
                  const int slot = b0 + __popc(m & ((1u << lane) - 1u));
                  if (slot < p.capg) {
                    p.cand_score[(int64_t)q * p.capg + slot] = agg;
                    p.cand_id[(int64_t)q * p.capg + slot] = doc;
                  } else {
                    p.overflow[q] = 1;
                  }
                }
              }
            }
            continue;
          }
          unsigned mym = 0;  // lane j: documents (lanes) passing column j
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const unsigned m = __ballot_sync(MEVI_FULL_MASK, (mk >> j) & 1u);
            if (lane == j) mym = m;
          }
          const int myq = qid[c0 + lane];
          int base_l = 0;
          if (mym && myq >= 0) base_l = atomicAdd(&p.count[myq], __popc(mym));
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int b0 = __shfl_sync(MEVI_FULL_MASK, base_l, j);
            const unsigned m = __shfl_sync(MEVI_FULL_MASK, mym, j);
            const int q = __shfl_sync(MEVI_FULL_MASK, myq, j);
            if (((mk >> j) & 1u) && q >= 0) {
              const int slot = b0 + __popc(m & ((1u << lane) - 1u));
              if (slot < p.capg) {
                p.cand_score[(int64_t)q * p.capg + slot] = __uint_as_float(acc[j]) * inv;
                p.cand_id[(int64_t)q * p.capg + slot] = doc;
              } else {
                p.overflow[q] = 1;  // per query: only this query is re-run through the streaming kernel
              }
            }
          }
        }
      }
      // the threshold / query-id slots of this buffer are rewritten two items later: every epilogue warp
      // passes the named barrier of the NEXT item before that, so no extra synchronisation is needed here
    }
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  if (warp == 0) ptx::tmem_dealloc(tmem_base, 2 * ACC_COLS);
}

// columns in use per group, rounded up to the UMMA N granule (the planners fill a group's columns from 0 upwards)
__global__ void gr_group_cols_kernel(const int32_t* __restrict__ group_qid, int64_t n_groups, int32_t* __restrict__ ncols) {
  const int lane = threadIdx.x & 31;
  const int64_t g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (g >= n_groups) return;
  const int q0 = group_qid[g * GR_TN + lane], q1 = group_qid[g * GR_TN + 32 + lane];
  const unsigned m0 = __ballot_sync(MEVI_FULL_MASK, q0 >= 0), m1 = __ballot_sync(MEVI_FULL_MASK, q1 >= 0);
  const int last = m1 ? 64 - __clz(m1) : (m0 ? 32 - __clz(m0) : 0);  // one past the last column in use
  if (lane == 0) ncols[g] = max(16, (last + 15) & ~15);
}

// the call's queries in fp16 (scaled by consts[FC_SQ], clamped like to_fp16_image_kernel), row-major: one warp per row
__global__ void gr_q16_kernel(const float* __restrict__ Q, int nq, int d, const float* __restrict__ consts,
                              __half* __restrict__ q16, int* __restrict__ clamped) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= nq) return;
  const float s = consts[FC_SQ];
  bool clamp = false;
  for (int u = lane; u < d / 8; u += 32) {
    const float4 a = ldg_f4(Q + (int64_t)row * d + u * 8), b = ldg_f4(Q + (int64_t)row * d + u * 8 + 4);
    const float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    __half h[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      float t = v[e] * s;
      if (fabsf(t) > 65000.f) { t = copysignf(65000.f, t); clamp = true; }
      h[e] = __float2half_rn(t);
    }
    *reinterpret_cast<uint4*>(q16 + (int64_t)row * d + u * 8) = *reinterpret_cast<const uint4*>(h);
  }
  if (clamp) atomicExch(clamped, 1);
}

// group images [group][K chunk][64 rows][64] (128B-swizzled as UMMA reads them) copied from the fp16 queries; only
// the rows in use (group_ncols) are written.  One CTA per group (grid-stride), one warp per row, two rows in flight.
__global__ void __launch_bounds__(256) gr_group_image_kernel(const __half* __restrict__ q16, int d,
                                                             const int32_t* __restrict__ group_qid,
                                                             const int32_t* __restrict__ group_ncols, int64_t n_groups,
                                                             __half* __restrict__ img) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int units = d / 8, nchunks = d / FT_KC;
  for (int64_t g = blockIdx.x; g < n_groups; g += gridDim.x) {
    const int ncols = group_ncols[g];
    for (int r0 = warp; r0 < ncols; r0 += 16) {
      const int r1 = r0 + 8;
      const int qa = group_qid[g * GR_TN + r0];
      const int qb = r1 < ncols ? group_qid[g * GR_TN + r1] : -1;
      for (int u0 = lane; u0 < units; u0 += 96) {
        uint4 va[3], vb[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          const int u = u0 + 32 * i;
          va[i] = make_uint4(0u, 0u, 0u, 0u);
          vb[i] = va[i];
          if (u < units) {
            if (qa >= 0) va[i] = __ldg(reinterpret_cast<const uint4*>(q16 + (int64_t)qa * d) + u);
            if (qb >= 0) vb[i] = __ldg(reinterpret_cast<const uint4*>(q16 + (int64_t)qb * d) + u);
          }
        }
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          const int u = u0 + 32 * i;
          if (u >= units) break;
          const int chunk = u / 8, uu = u & 7;
          __half* base = img + ((size_t)g * nchunks + chunk) * GR_TN * FT_KC;
          *reinterpret_cast<uint4*>(base + (size_t)r0 * FT_KC + ((uu ^ (r0 & 7)) * 8)) = va[i];
          if (r1 < ncols) *reinterpret_cast<uint4*>(base + (size_t)r1 * FT_KC + ((uu ^ (r1 & 7)) * 8)) = vb[i];
        }
      }
    }
  }
}

template <int MAXG, bool MC>
int gr_launch(mevi_ctx* ctx, const GroupedParams& p, int grid, cudaStream_t st) {
  const size_t smem = (size_t)gr_stages(MAXG) * gr_stage_bytes(MAXG) + 2 * MAXG * GR_TN * 8 +
                      (2 * gr_stages(MAXG) + 4) * 8 + 16 + 1024;
  MEVI_CUDA(ctx, cudaFuncSetAttribute(grouped_gemm_kernel<MAXG, MC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  grouped_gemm_kernel<MAXG, MC><<<grid, GR_THREADS, smem, st>>>(p);
  return MEVI_OK;
}

template <bool MC>
int gr_launch_maxg(mevi_ctx* ctx, const GroupedParams& p, int maxg, int grid, cudaStream_t st) {
  return maxg == 1 ? gr_launch<1, MC>(ctx, p, grid, st) : (maxg == 2 ? gr_launch<2, MC>(ctx, p, grid, st) : gr_launch<4, MC>(ctx, p, grid, st));
}

__global__ void gr_set_u32_kernel(unsigned* p, unsigned v) { *p = v; }
__global__ void gr_count_failed_kernel(const int* __restrict__ ovq, int nq, int* out) {
  __shared__ int s_n;
  if (threadIdx.x == 0) s_n = 0;
  __syncthreads();
  int c = 0;
  for (int i = threadIdx.x; i < nq; i += blockDim.x) c += ovq[i] != 0;
  if (c) atomicAdd(&s_n, c);
  __syncthreads();
  if (threadIdx.x == 0) *out = s_n;
}
inline unsigned gr_f32_bits(float f) {
  unsigned u;
  memcpy(&u, &f, 4);
  return u;
}

__global__ void gr_row_norm_kernel(const float* __restrict__ X, int rows, int d, float* __restrict__ norms) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  float a = 0.f;
  for (int c = lane * 4; c < d; c += 128) {
    const float4 v = ldg_f4(X + (int64_t)row * d + c);
    a = fmaf(v.x, v.x, a); a = fmaf(v.y, v.y, a); a = fmaf(v.z, v.z, a); a = fmaf(v.w, v.w, a);
  }
  a = warp_sum(a);
  if (lane == 0) norms[row] = sqrtf(a);
}

__global__ void gr_init_kernel(float* tau, const float* tau0, int* count, int* flags, int* ovq, int nq) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nq) {
    const float t = tau0 ? tau0[i] : -CUDART_INF_F;
    tau[i] = (t == t) ? t : -CUDART_INF_F;
    count[i] = 0;
    ovq[i] = 0;
  }
  if (i < 4) flags[i] = 0;
}

struct GrState {
  float* consts; unsigned* absmax; int* flags; float* tau; float* margin; float* qnorm; int* count;
  float* cand_score; int32_t* cand_id;
  int* ovq;  // [nq] 1 = the guarantee could not be established for this query (buffer or margin-window overflow)
  __half* q16;  // [nq][d] the call's queries, scaled and rounded to fp16 once (_begin); the rounds' group images copy rows
};

// the per-call state lives in one scratch slot from _begin to _finish (same layout recomputed by each entry point)
bool gr_state(mevi_ctx* ctx, int nq, int d, GrState* s) {
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = (off + bytes + 255) & ~size_t(255); return o; };
  const size_t o_consts = take(FC_NUM * 4), o_abs = take(16), o_flags = take(16), o_tau = take((size_t)nq * 4),
               o_margin = take((size_t)nq * 4), o_qnorm = take((size_t)nq * 4), o_cnt = take((size_t)nq * 4),
               o_ovq = take((size_t)nq * 4), o_cs = take((size_t)nq * GR_CAPG * 4), o_ci = take((size_t)nq * GR_CAPG * 4),
               o_q16 = take((size_t)nq * d * 2);
  char* ws = (char*)mevi_ws(ctx, WS_TOPK_AUX, off);
  if (!ws) return false;
  s->consts = (float*)(ws + o_consts); s->absmax = (unsigned*)(ws + o_abs); s->flags = (int*)(ws + o_flags);
  s->tau = (float*)(ws + o_tau); s->margin = (float*)(ws + o_margin); s->qnorm = (float*)(ws + o_qnorm);
  s->count = (int*)(ws + o_cnt); s->cand_score = (float*)(ws + o_cs); s->cand_id = (int32_t*)(ws + o_ci);
  s->ovq = (int*)(ws + o_ovq);
  s->q16 = (__half*)(ws + o_q16);
  return true;
}

// ---- multi-cluster call state (mevi_rerank_grouped_multiclus .. _finish_multiclus) ----
struct GrMcHost {  // plain data: lives in mevi_ctx::gr_mc
  int valid, nq, qtab_log2, C, aggr;
  const int32_t* occ; const int32_t* tile_leaf; const int64_t* leaf_offsets; int64_t n_leaves;
};
struct GrMcState { uint64_t* qtab; float* cheap; float* m_mc; };

bool gr_mc_state(mevi_ctx* ctx, int nq, int log2, GrMcState* s) {
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = (off + bytes + 255) & ~size_t(255); return o; };
  const size_t o_tab = take((size_t)nq * (8u << log2)), o_cheap = take((size_t)nq * 4), o_m = take((size_t)nq * 4);
  char* ws = (char*)mevi_ws(ctx, WS_GR_MC, off);
  if (!ws) return false;
  s->qtab = (uint64_t*)(ws + o_tab); s->cheap = (float*)(ws + o_cheap); s->m_mc = (float*)(ws + o_m);
  return true;
}

// the attached multi-cluster state of the current call, or nullptr (a single-cluster call)
const GrMcHost* gr_mc_attached(mevi_ctx* ctx, int nq) {
  const GrMcHost* h = (const GrMcHost*)ctx->gr_mc;
  return h && h->valid && h->nq == nq ? h : nullptr;
}

// One CTA per query: its leaf table (from the UNMASKED list: c counts every position), n_candidates (every position, like
// the streaming kernel), the list with every later position of a repeated leaf set to -1 (one plan pair per distinct leaf),
// and from c_max = C x the largest repetition of a leaf (an upper bound of c):
//   m_mc = c_max margin + c_max (c_max - 1) 2^-24 (4.05 |q| dmax + 1.01 margin),  x (1 + 2^-13) for its own fp32 evaluation
//   cheap = 1 / (c_max (1 + (c_max + 4) 2^-21))
// ('max': m_mc = margin, cheap = 1).  DESIGN §4 derives both.
__global__ void __launch_bounds__(256) gr_mc_table_kernel(const int32_t* __restrict__ ql, int L, const int64_t* __restrict__ off,
                                                          int64_t n_leaves, int C, int aggr, int log2, const float* __restrict__ margin,
                                                          const float* __restrict__ qnorm, const unsigned* __restrict__ dmax_bits,
                                                          uint64_t* __restrict__ qtab, float* __restrict__ cheap,
                                                          float* __restrict__ m_mc, int32_t* __restrict__ ql_masked,
                                                          int32_t* __restrict__ ncand) {
  extern __shared__ int32_t s_tab[];  // key | first position | number of positions, [1 << log2] each
  const int H = 1 << log2;
  int32_t* s_key = s_tab;
  int32_t* s_first = s_tab + H;
  int32_t* s_mult = s_tab + 2 * H;
  __shared__ long long s_tot[8];
  __shared__ int s_rep[8];
  const int q = blockIdx.x, tid = threadIdx.x;
  for (int i = tid; i < H; i += blockDim.x) { s_key[i] = -1; s_first[i] = 0x7fffffff; s_mult[i] = 0; }
  __syncthreads();
  long long tot = 0;
  for (int t = tid; t < L; t += blockDim.x) {
    const int leaf = ql[(int64_t)q * L + t];
    if (leaf < 0 || leaf >= n_leaves) continue;
    const int64_t sz = off[leaf + 1] - off[leaf];
    tot += sz;
    if (sz == 0) continue;  // no document: never scored, never a sibling
    const unsigned mask = (unsigned)H - 1u;
    unsigned h = ((unsigned)leaf * 0x9E3779B1u) >> (32 - log2);
    for (;;) {
      const int prev = atomicCAS(&s_key[h], -1, leaf);
      if (prev < 0 || prev == leaf) break;
      h = (h + 1) & mask;
    }
    atomicMin(&s_first[h], t);
    atomicAdd(&s_mult[h], 1);
  }
  __syncthreads();
  int rep = 0;
  for (int t = tid; t < L; t += blockDim.x) {
    const int leaf = ql[(int64_t)q * L + t];
    int keep = -1;
    if (leaf >= 0 && leaf < n_leaves && off[leaf + 1] > off[leaf]) {
      unsigned h = ((unsigned)leaf * 0x9E3779B1u) >> (32 - log2);
      while (s_key[h] != leaf) h = (h + 1) & ((unsigned)H - 1u);
      if (s_first[h] == t) keep = leaf;
    }
    ql_masked[(int64_t)q * L + t] = keep;
  }
  for (int i = tid; i < H; i += blockDim.x) {
    const int k = s_key[i];
    qtab[(int64_t)q * H + i] = k < 0 ? ~0ull : ((uint64_t)(uint32_t)k | ((uint64_t)s_first[i] << 32) | ((uint64_t)s_mult[i] << 48));
    rep = max(rep, s_mult[i]);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    tot += __shfl_xor_sync(MEVI_FULL_MASK, tot, o);
    rep = max(rep, __shfl_xor_sync(MEVI_FULL_MASK, rep, o));
  }
  if ((tid & 31) == 0) { s_tot[tid >> 5] = tot; s_rep[tid >> 5] = rep; }
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) { tot += s_tot[w]; rep = max(rep, s_rep[w]); }
    ncand[q] = (int32_t)(tot > 0x7FFFFFFFll ? 0x7FFFFFFFll : tot);
    const float cm = (float)max(C * rep, 1), mq = margin[q];
    if (aggr == MEVI_MULTICLUS_ADD) {
      const float B = qnorm[q] * __uint_as_float(*dmax_bits);
      m_mc[q] = (cm * mq + cm * (cm - 1.f) * 5.9604645e-8f * (4.05f * B + 1.01f * mq)) * 1.0001221f;
      cheap[q] = 1.f / (cm * (1.f + (cm + 4.f) * 4.7683716e-7f));
    } else {
      m_mc[q] = mq;
      cheap[q] = 1.f;
    }
  }
}

// flat_rescore_kernel for a multi-cluster call: the same exact re-score (the dense scorer's summation order, as the
// streaming kernel), then c from the query's leaf table and the fold; sorted by (aggregated score desc, DOCUMENT id asc):
// leaf order is not document order when documents sit under several leaves.  ids = id_base + leaf_docids[row].
__global__ void __launch_bounds__(256) gr_mc_rescore_kernel(const float* __restrict__ Q, const float* __restrict__ D, int d,
                                                            const int* __restrict__ count, const int32_t* __restrict__ cand_id,
                                                            const float* __restrict__ cand_score, const float* __restrict__ tau,
                                                            const float* __restrict__ margin, int capg, int k, int keep_pow2,
                                                            const int64_t* __restrict__ off, int64_t n_leaves,
                                                            const int32_t* __restrict__ occ, int occ_w,
                                                            const uint64_t* __restrict__ qtab, int log2, int aggr,
                                                            const int32_t* __restrict__ leaf_docids, int64_t id_base,
                                                            float* __restrict__ scores, int64_t* __restrict__ ids) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* s_score = reinterpret_cast<float*>(smem_raw);
  int32_t* s_id = reinterpret_cast<int32_t*>(s_score + keep_pow2);
  const int q = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int cnt = count[q];
  if (cnt > keep_pow2) cnt = keep_pow2;
  for (int i = threadIdx.x; i < keep_pow2; i += blockDim.x) {
    s_score[i] = -CUDART_INF_F;
    s_id[i] = 0x7fffffff;
  }
  __syncthreads();
  const float window = tau[q] - margin[q];
  for (int i = warp; i < cnt; i += 8) {
    if (cand_score[(int64_t)q * capg + i] < window) continue;
    const int32_t row = cand_id[(int64_t)q * capg + i];
    float acc = 0.f;
    for (int c4 = lane * 4; c4 < d; c4 += 128) {  // same summation pattern as the dense scorer
      const float4 a = ldg_f4(Q + (int64_t)q * d + c4);
      const float4 b = ld_stream_f4(D + (int64_t)row * d + c4);
      acc = fmaf(a.x, b.x, acc);
      acc = fmaf(a.y, b.y, acc);
      acc = fmaf(a.z, b.z, acc);
      acc = fmaf(a.w, b.w, acc);
    }
    acc = warp_sum(acc);
    if (lane == 0) {
      if (aggr == MEVI_MULTICLUS_ADD) {
        int64_t lo = 0, hi = n_leaves;  // leaf of the row: last leaf whose first row is <= row
        while (hi - lo > 1) {
          const int64_t mid = (lo + hi) >> 1;
          if (off[mid] <= row) lo = mid; else hi = mid;
        }
        // every kept occurrence is canonical, so c >= 1
        acc = mc_fold(acc, mc_count(qtab + ((int64_t)q << log2), log2, (int)lo, occ + (int64_t)row * occ_w, occ_w));
      }
      s_score[i] = acc;
      s_id[i] = leaf_docids[row];
    }
  }
  __syncthreads();
  block_bitonic_sort<int32_t>(s_score, s_id, keep_pow2);
  for (int i = threadIdx.x; i < k; i += blockDim.x) {
    const bool ok = i < cnt && s_id[i] != 0x7fffffff;
    scores[(int64_t)q * k + i] = ok ? s_score[i] : -CUDART_INF_F;
    ids[(int64_t)q * k + i] = ok ? id_base + (int64_t)s_id[i] : -1;
  }
}

}  // namespace

// fp16 image of the leaf-ordered matrix, tiles of 128 rows that never straddle a leaf.
//   src_index [n_tiles*128] int32: row of D_leaf for every image row, -1 = padding
//   absmax_out / maxnorm_out (host): the two numbers _begin needs (scale of the image, largest document norm)
extern "C" int mevi_rerank_grouped_image(mevi_ctx* ctx, const float* D_leaf, int64_t n, int d, const int32_t* src_index,
                                         int64_t n_tiles, void* Aimg, float* absmax_out, float* maxnorm_out, void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  MEVI_REQUIRE(ctx, D_leaf && src_index && Aimg && absmax_out && maxnorm_out, "NULL argument");
  MEVI_REQUIRE(ctx, mevi_flat_tensor_supported(ctx, d, 1), "grouped re-rank needs sm_100 and d %% 64 == 0 (got d=%d)", d);
  MEVI_REQUIRE(ctx, n > 0 && n < (int64_t)2147483647 && n_tiles > 0, "bad sizes");
  char* ws = (char*)mevi_ws(ctx, WS_MISC, 512);
  if (!ws) return MEVI_ERR_NOMEM;
  float* consts = (float*)ws;                 // FC_NUM floats
  unsigned* absmax2 = (unsigned*)(ws + 64);   // [0] D absmax, [1] unused (1.0), [2] max doc norm
  int* flags = (int*)(ws + 128);
  MEVI_CUDA(ctx, cudaMemsetAsync(ws, 0, 512, st));
  const int64_t sample_rows = 4096;
  flat_absmax_kernel<<<ctx->sm_count, 256, 0, st>>>(D_leaf, n, d, n > sample_rows ? n / sample_rows : 1, absmax2);
  gr_set_u32_kernel<<<1, 1, 0, st>>>(absmax2 + 1, gr_f32_bits(1.0f));
  gr_consts_kernel<<<1, 32, 0, st>>>(absmax2, consts);
  to_fp16_image_kernel<<<ctx->sm_count * 8, 256, 0, st>>>(D_leaf, n, d, FT_TM, consts, FC_SD, (__half*)Aimg, nullptr, absmax2 + 2,
                                                          flags, n_tiles * FT_TM, src_index);
  MEVI_CUDA(ctx, cudaGetLastError());
  MEVI_COUNT_LAUNCH(ctx, 4);
  unsigned h[4] = {0, 0, 0, 0};
  int h_flag = 0;
  MEVI_CUDA(ctx, cudaMemcpyAsync(h, absmax2, sizeof(h), cudaMemcpyDeviceToHost, st));
  MEVI_CUDA(ctx, cudaMemcpyAsync(&h_flag, flags, sizeof(int), cudaMemcpyDeviceToHost, st));
  MEVI_CUDA(ctx, cudaStreamSynchronize(st));
  if (int drc = mevi_deferred_error(ctx)) return drc;  // a kernel of this (or an earlier asynchronous) launch timed out
  float a, m;
  memcpy(&a, &h[0], 4);
  memcpy(&m, &h[2], 4);
  *absmax_out = h_flag ? -1.f : a;  // a clamped image cannot carry the guarantee: the caller keeps the streaming kernel
  *maxnorm_out = m;
  return MEVI_OK;
}

// start of a grouped re-rank call: query scale / norms / margins, thresholds from tau0 (device, may be NULL)
extern "C" int mevi_rerank_grouped_begin(mevi_ctx* ctx, const float* Q, int nq, int d, float d_absmax, float d_maxnorm,
                                         const float* tau0, void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  MEVI_REQUIRE(ctx, Q && nq > 0 && d_absmax >= 0.f, "bad argument");
  GrState s;
  if (!gr_state(ctx, nq, d, &s)) return MEVI_ERR_NOMEM;
  if (ctx->gr_mc) ((GrMcHost*)ctx->gr_mc)->valid = 0;  // a new call: single-cluster unless _multiclus attaches its state
  gr_init_kernel<<<(nq + 255) / 256, 256, 0, st>>>(s.tau, tau0, s.count, s.flags, s.ovq, nq);
  gr_set_u32_kernel<<<1, 1, 0, st>>>(s.absmax + 0, gr_f32_bits(d_absmax));
  gr_set_u32_kernel<<<1, 1, 0, st>>>(s.absmax + 1, 0u);
  gr_set_u32_kernel<<<1, 1, 0, st>>>(s.absmax + 2, gr_f32_bits(d_maxnorm));
  flat_absmax_kernel<<<ctx->sm_count, 256, 0, st>>>(Q, nq, d, 1, s.absmax + 1);
  gr_consts_kernel<<<1, 32, 0, st>>>(s.absmax, s.consts);
  gr_row_norm_kernel<<<(nq + 7) / 8, 256, 0, st>>>(Q, nq, d, s.qnorm);
  flat_margin_kernel<<<(nq + 255) / 256, 256, 0, st>>>(s.qnorm, nq, d, s.absmax + 2, s.consts, s.margin);
  gr_q16_kernel<<<(nq + 7) / 8, 256, 0, st>>>(Q, nq, d, s.consts, s.q16, s.flags + 2);
  MEVI_CUDA(ctx, cudaGetLastError());
  MEVI_COUNT_LAUNCH(ctx, 9);
  return MEVI_OK;
}

// one round: gather the query image of the round's groups, run the grouped GEMM, tighten the thresholds
extern "C" int mevi_rerank_grouped_round(mevi_ctx* ctx, const float* Q, int nq, int d, const void* Aimg,
                                         const int32_t* tile_row0, const int32_t* tile_nrows, const int32_t* item_tile,
                                         const int32_t* item_group, int64_t n_items, const int32_t* group_qid,
                                         int64_t n_groups, int max_groups_per_item, int k, void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  MEVI_REQUIRE(ctx, Q && Aimg && tile_row0 && tile_nrows, "NULL argument");
  MEVI_REQUIRE(ctx, k >= 1 && k <= FT_KEEP / 2, "k must be in [1, %d]", FT_KEEP / 2);
  if (n_items <= 0 || n_groups <= 0) return MEVI_OK;
  MEVI_REQUIRE(ctx, item_tile && item_group && group_qid, "NULL argument");
  MEVI_REQUIRE(ctx, max_groups_per_item >= 1 && max_groups_per_item <= 4 && n_groups <= (int64_t)GR_GROUP_MASK,
               "items take 1..4 groups and a round at most %u groups", GR_GROUP_MASK);
  GrState s;
  if (!gr_state(ctx, nq, d, &s)) return MEVI_ERR_NOMEM;
  const int nchunks = d / FT_KC;
  const size_t img_bytes = ((size_t)n_groups * GR_TN * d * 2 + 255) & ~size_t(255);
  char* bws = (char*)mevi_ws(ctx, WS_TOPK_PART, img_bytes + (size_t)n_groups * 4);
  if (!bws) return MEVI_ERR_NOMEM;
  __half* Bimg = (__half*)bws;
  int32_t* group_ncols = (int32_t*)(bws + img_bytes);
  gr_group_cols_kernel<<<(unsigned)((n_groups + 7) / 8), 256, 0, st>>>(group_qid, n_groups, group_ncols);
  gr_group_image_kernel<<<(unsigned)(n_groups < (int64_t)ctx->sm_count * 8 ? n_groups : (int64_t)ctx->sm_count * 8), 256, 0, st>>>(
      s.q16, d, group_qid, group_ncols, n_groups, Bimg);
  GroupedParams p;
  p.Aimg = (const __half*)Aimg; p.Bimg = Bimg; p.item_tile = item_tile; p.item_group = item_group; p.n_items = n_items;
  p.tile_row0 = tile_row0; p.tile_nrows = tile_nrows; p.group_qid = group_qid; p.group_ncols = group_ncols; p.nchunks = nchunks;
  p.consts = s.consts; p.tau = s.tau; p.margin = s.margin; p.count = s.count; p.cand_score = s.cand_score;
  p.cand_id = s.cand_id; p.overflow = s.ovq; p.capg = GR_CAPG; p.err_flag = s.flags + 1;
  p.occ = nullptr; p.occ_w = 0; p.tile_leaf = nullptr; p.qtab = nullptr; p.qtab_log2 = 1; p.mc_cheap = nullptr; p.aggr = 0;
  const GrMcHost* mc = gr_mc_attached(ctx, nq);
  if (mc) {  // multi-cluster call: the MC epilogue, and the aggregated margin for it and for the compaction
    GrMcState ms;
    if (!gr_mc_state(ctx, nq, mc->qtab_log2, &ms)) return MEVI_ERR_NOMEM;
    p.margin = ms.m_mc; p.occ = mc->occ; p.occ_w = mc->C - 1; p.tile_leaf = mc->tile_leaf; p.qtab = ms.qtab;
    p.qtab_log2 = mc->qtab_log2; p.mc_cheap = ms.cheap; p.aggr = mc->aggr;
  }
  const int grid = (int)(n_items < ctx->sm_count ? n_items : ctx->sm_count);
  const int maxg = max_groups_per_item <= 1 ? 1 : (max_groups_per_item == 2 ? 2 : 4);
  if (int rc = mc ? gr_launch_maxg<true>(ctx, p, maxg, grid, st) : gr_launch_maxg<false>(ctx, p, maxg, grid, st)) return rc;
  const size_t smem_compact = (size_t)GR_CAPG * 8;
  MEVI_CUDA(ctx, cudaFuncSetAttribute(flat_tensor_compact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_compact));
  flat_tensor_compact_kernel<<<nq, 256, smem_compact, st>>>(s.tau, p.margin, s.count, s.cand_score, s.cand_id, s.ovq, GR_CAPG, k,
                                                            FT_KEEP, 1);
  MEVI_CUDA(ctx, cudaGetLastError());
  MEVI_COUNT_LAUNCH(ctx, 4);
  return MEVI_OK;
}

// thresholds of the call between rounds: raise == 0 copies them out, raise != 0 lifts them to max(own, given).  With the
// documents sharded over ranks, max over ranks of the local k-th best scores is a lower bound of the global k-th best:
// an all-reduce(MAX) between the two calls lets every rank filter (and finally re-score) against the global bound.
__global__ void gr_raise_tau_kernel(float* __restrict__ tau, const float* __restrict__ given, int nq) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nq) tau[i] = fmaxf(tau[i], given[i]);
}

extern "C" int mevi_rerank_grouped_thresholds(mevi_ctx* ctx, int nq, int d, float* tau, int raise, void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  MEVI_REQUIRE(ctx, tau && nq > 0 && d > 0, "bad argument");
  GrState s;
  if (!gr_state(ctx, nq, d, &s)) return MEVI_ERR_NOMEM;
  if (raise) {
    gr_raise_tau_kernel<<<(nq + 255) / 256, 256, 0, st>>>(s.tau, tau, nq);
    MEVI_CUDA(ctx, cudaGetLastError());
    MEVI_COUNT_LAUNCH(ctx, 1);
  } else {
    MEVI_CUDA(ctx, cudaMemcpyAsync(tau, s.tau, (size_t)nq * sizeof(float), cudaMemcpyDeviceToDevice, st));
  }
  return MEVI_OK;
}

// end of the call.  *n_failed = nq when the whole call is invalid (a query element left the fp16 range): the caller runs
// the streaming kernel.  Otherwise scores [nq,k] fp32 descending and rows [nq,k] int64 = rows of the leaf-ordered matrix
// (-1 padded), *n_failed = number of queries whose guarantee could not be established (candidate buffer or margin window
// overflow: near-duplicate documents, one huge leaf) and failed_or_null [nq] (device, int32) marks them: the caller
// re-runs just those through mevi_cluster_rerank.
namespace {
// _finish and _finish_multiclus (mc != nullptr: rows -> document ids, see gr_mc_rescore_kernel)
int gr_finish(mevi_ctx* ctx, const float* Q, int nq, const float* D_leaf, int d, int k, const GrMcHost* mc,
              const int32_t* leaf_docids, int64_t id_base, float* scores, int64_t* rows, int32_t* failed_or_null, int* n_failed,
              cudaStream_t st) {
  *n_failed = nq;
  GrState s;
  if (!gr_state(ctx, nq, d, &s)) return MEVI_ERR_NOMEM;
  int h_flags[4] = {0, 0, 0, 0};
  gr_count_failed_kernel<<<1, 256, 0, st>>>(s.ovq, nq, s.flags + 3);
  MEVI_COUNT_LAUNCH(ctx, 1);
  if (failed_or_null) MEVI_CUDA(ctx, cudaMemcpyAsync(failed_or_null, s.ovq, (size_t)nq * sizeof(int), cudaMemcpyDeviceToDevice, st));
  MEVI_CUDA(ctx, cudaMemcpyAsync(h_flags, s.flags, sizeof(h_flags), cudaMemcpyDeviceToHost, st));
  MEVI_CUDA(ctx, cudaStreamSynchronize(st));
  if (int drc = mevi_deferred_error(ctx)) return drc;  // a kernel of this (or an earlier asynchronous) launch timed out
  if (h_flags[1]) return mevi_set_error(ctx, MEVI_ERR_CUDA, "grouped re-rank pipeline time-out (code %d)", h_flags[1]);
  if (h_flags[2]) return MEVI_OK;  // clamped query image: nothing of this call carries the guarantee
  const size_t smem_rescore = (size_t)FT_KEEP * 8;
  if (mc) {
    GrMcState ms;
    if (!gr_mc_state(ctx, nq, mc->qtab_log2, &ms)) return MEVI_ERR_NOMEM;
    gr_mc_rescore_kernel<<<nq, 256, smem_rescore, st>>>(Q, D_leaf, d, s.count, s.cand_id, s.cand_score, s.tau, ms.m_mc, GR_CAPG, k,
                                                        FT_KEEP, mc->leaf_offsets, mc->n_leaves, mc->occ, mc->C - 1, ms.qtab,
                                                        mc->qtab_log2, mc->aggr, leaf_docids, id_base, scores, rows);
  } else {
    flat_rescore_kernel<<<nq, 256, smem_rescore, st>>>(Q, D_leaf, d, s.count, s.cand_id, s.cand_score, s.tau, s.margin, GR_CAPG, k,
                                                       FT_KEEP, 0, scores, rows);
  }
  MEVI_CUDA(ctx, cudaGetLastError());
  MEVI_COUNT_LAUNCH(ctx, 1);
  *n_failed = h_flags[3];
  return MEVI_OK;
}
}  // namespace

extern "C" int mevi_rerank_grouped_finish(mevi_ctx* ctx, const float* Q, int nq, const float* D_leaf, int d, int k,
                                          float* scores, int64_t* rows, int32_t* failed_or_null, int* n_failed, void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  MEVI_REQUIRE(ctx, Q && D_leaf && scores && rows && n_failed, "NULL argument");
  return gr_finish(ctx, Q, nq, D_leaf, d, k, nullptr, nullptr, 0, scores, rows, failed_or_null, n_failed, (cudaStream_t)stream);
}

// Multi-cluster index (--doc_multiclus > 1): attach the call's multi-cluster state after _begin; _round then runs the MC
// epilogue and _finish_multiclus ends the call.
extern "C" int mevi_rerank_grouped_multiclus(mevi_ctx* ctx, int nq, int d, const int32_t* query_leaves, int L,
                                             const int64_t* leaf_offsets, int64_t n_leaves, const int32_t* occ_leaves, int C,
                                             const int32_t* tile_leaf, int aggr, int32_t* query_leaves_masked,
                                             int32_t* n_candidates, void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  MEVI_REQUIRE(ctx, query_leaves && leaf_offsets && tile_leaf && query_leaves_masked && n_candidates, "NULL argument");
  MEVI_REQUIRE(ctx, nq > 0 && d > 0 && L > 0 && n_leaves > 0, "bad extents");
  MEVI_REQUIRE(ctx, aggr == MEVI_MULTICLUS_ADD || aggr == MEVI_MULTICLUS_MAX, "aggr must be MEVI_MULTICLUS_ADD or _MAX (got %d)", aggr);
  MEVI_REQUIRE(ctx, C >= 1 && (C == 1 || occ_leaves), "C must be >= 1, with an occurrence table when C > 1");
  if (C > 16 || L > 4096)
    return mevi_set_error(ctx, MEVI_ERR_UNSUPPORTED, "grouped multi-cluster re-rank: C = %d (at most 16), L = %d (at most 4096)", C, L);
  GrState s;
  if (!gr_state(ctx, nq, d, &s)) return MEVI_ERR_NOMEM;
  int log2 = 1;
  while ((1 << log2) < 2 * L) ++log2;
  GrMcState ms;
  if (!gr_mc_state(ctx, nq, log2, &ms)) return MEVI_ERR_NOMEM;
  if (!ctx->gr_mc) ctx->gr_mc = calloc(1, sizeof(GrMcHost));
  if (!ctx->gr_mc) return mevi_set_error(ctx, MEVI_ERR_NOMEM, "grouped multi-cluster re-rank: host state");
  const size_t smem = (size_t)12 << log2;
  MEVI_CUDA(ctx, cudaFuncSetAttribute(gr_mc_table_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  gr_mc_table_kernel<<<nq, 256, smem, st>>>(query_leaves, L, leaf_offsets, n_leaves, C, aggr, log2, s.margin, s.qnorm, s.absmax + 2,
                                            ms.qtab, ms.cheap, ms.m_mc, query_leaves_masked, n_candidates);
  MEVI_CUDA(ctx, cudaGetLastError());
  MEVI_COUNT_LAUNCH(ctx, 1);
  GrMcHost& h = *(GrMcHost*)ctx->gr_mc;
  h.nq = nq; h.qtab_log2 = log2; h.C = C; h.aggr = aggr; h.occ = C > 1 ? occ_leaves : nullptr; h.tile_leaf = tile_leaf;
  h.leaf_offsets = leaf_offsets; h.n_leaves = n_leaves;
  h.valid = 1;
  return MEVI_OK;
}

extern "C" int mevi_rerank_grouped_finish_multiclus(mevi_ctx* ctx, const float* Q, int nq, const float* D_leaf, int d, int k,
                                                    const int32_t* leaf_docids, int64_t id_base, float* scores, int64_t* ids,
                                                    int32_t* failed_or_null, int* n_failed, void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  MEVI_REQUIRE(ctx, Q && D_leaf && leaf_docids && scores && ids && n_failed, "NULL argument");
  const GrMcHost* mc = gr_mc_attached(ctx, nq);
  MEVI_REQUIRE(ctx, mc, "no multi-cluster state: call mevi_rerank_grouped_multiclus after _begin");
  const int rc = gr_finish(ctx, Q, nq, D_leaf, d, k, mc, leaf_docids, id_base, scores, ids, failed_or_null, n_failed,
                           (cudaStream_t)stream);
  ((GrMcHost*)ctx->gr_mc)->valid = 0;
  return rc;
}


// =====================================================================================================
// Persistent flat index: faiss `index.add(doc)` once, `index.search(query, k)` many (faiss_search.py:15-20).
// The fp16 tile image and the document-side metadata are built by _create and owned by the index; D itself stays
// caller-owned and must outlive the index (the exact re-score and the fp32 fall-back read it).
struct mevi_flat_index {
  const float* D;
  int64_t n;
  int d;
  __half* Aimg;       // nullptr: shape outside the tensor path, searches run the fp32 kernel
  unsigned* docmeta;  // DM_NUM words
};

extern "C" int mevi_flat_index_create(mevi_ctx* ctx, const float* D, int64_t n, int d, mevi_flat_index** out, void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  MEVI_REQUIRE(ctx, out && (D || n == 0) && n >= 0 && d > 0, "bad argument");
  MEVI_REQUIRE(ctx, n < (int64_t)2147483647, "index too large for int32 row ids (shard it)");
  *out = nullptr;
  mevi_flat_index* ix = new mevi_flat_index{D, n, d, nullptr, nullptr};
  if (n > 0 && mevi_flat_tensor_supported(ctx, d, 1) && (reinterpret_cast<uintptr_t>(D) & 15) == 0) {
    const int64_t n_tiles = (n + FT_TM - 1) / FT_TM;
    if (cudaMalloc(&ix->Aimg, (size_t)n_tiles * FT_TM * d * 2) != cudaSuccess || cudaMalloc(&ix->docmeta, 256) != cudaSuccess) {
      cudaGetLastError();
      if (ix->Aimg) cudaFree(ix->Aimg);
      delete ix;
      return mevi_set_error(ctx, MEVI_ERR_NOMEM, "flat index: cudaMalloc of the %lld-row fp16 image failed", (long long)n);
    }
    const int rc = flat_docs_prepare(ctx, D, n, d, ix->Aimg, ix->docmeta, st);
    if (rc != MEVI_OK) {
      cudaFree(ix->Aimg);
      cudaFree(ix->docmeta);
      delete ix;
      return rc;
    }
  }
  *out = ix;
  return MEVI_OK;
}

extern "C" int mevi_flat_index_search(mevi_ctx* ctx, const mevi_flat_index* ix, const float* Q, int nq, int k, int64_t id_base,
                                      int mode, float* scores, int64_t* ids, void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  MEVI_REQUIRE(ctx, ix && scores && ids && (Q || nq == 0), "NULL argument");
  if (nq <= 0) return MEVI_OK;
  if (ix->Aimg != nullptr && mevi_flat_tensor_supported(ctx, ix->d, k) &&
      (mode == MEVI_MODE_TENSOR || (mode == MEVI_MODE_AUTO && ix->n >= 8192))) {
    int fell_back = 1;
    const int rc = mevi_flat_tensor_search_image(ctx, Q, nq, ix->D, ix->n, ix->d, ix->Aimg, ix->docmeta, k, id_base, scores, ids,
                                                 &fell_back, st);
    if (rc != MEVI_OK) return rc;
    if (!fell_back) return MEVI_OK;
  } else if (mode == MEVI_MODE_TENSOR) {
    return mevi_set_error(ctx, MEVI_ERR_UNSUPPORTED, "tensor flat search unsupported for this index (d=%d k=%d n=%lld)", ix->d, k,
                          (long long)ix->n);
  }
  return mevi_flat_ip_topk(ctx, Q, nq, ix->D, ix->n, ix->d, k, id_base, MEVI_MODE_EXACT, scores, ids, stream);
}

extern "C" void mevi_flat_index_destroy(mevi_ctx* ctx, mevi_flat_index* ix) {
  if (!ix) return;
  if (ctx) {
    DeviceGuard g(ctx->device);
    cudaDeviceSynchronize();
    if (ix->Aimg) cudaFree(ix->Aimg);
    if (ix->docmeta) cudaFree(ix->docmeta);
  }
  delete ix;
}
