// pq_tensor.cuh — product-quantiser encode on the tensor cores for the wide codebooks (K = 256 centroids per
// sub-vector, sub-vector width 32 or 24: 24 x 256 and the reference default 32 x 256 at d = 768).  Replaces MEVI/pq.py:249-279 for
// those shapes; the M*K <= 128 shapes ride on K1 (pq_encode.cu), everything else on the fp32 sub-vector kernel.
//
// Per sub-vector j the scores  s_k = 2 x_j.c_k - |c_k|^2  ('l2': the reference's -|x_j - c_k|^2 up to the row constant)
// or  x_j.c_k  ('ip') of 256 centroids are one [rows x 32] . [32 x 256] contraction: split-fp16 (hi.hi + hi.lo + lo.hi,
// ~2^-22 relative) on tcgen05 with the document operand in TENSOR MEMORY, as in K1 generation 4.  What differs from K1:
//   * the codebook operand of a sub-vector is 48 KB (K1: 16 KB per chunk for all levels), so it cannot be streamed per
//     row tile.  The CTA keeps the images of THREE sub-vectors (144 KB) resident and walks ALL its row tiles for them,
//     then loads the next three: the document matrix is still read exactly once, in passes over 384-byte row pieces;
//   * a unit of work is (128 rows, sub-vector, half of the centroids): N = 128 accumulator columns, THREE buffers in
//     rotation (unit u -> buffer u % 3) so the MMAs of the next unit run while two units are being drained; MMA warp h
//     issues the units of half h (two independent issue streams fill each other's commit bubbles);
//   * the epilogue reduces 256 scores per (row, sub-vector) - 6,144 per row - and is the issue-bound part of the
//     kernel (K = 32 per accumulator: an epilogue-heavy GEMM), so everything that can leave it has left it:
//       - the -|c_k|^2 term rides on the tensor cores: a 7th MMA per unit multiplies a constant operand tile (2^8 in
//         three K slots) with a third codebook block holding -|c_k|^2 (in accumulator units, / 2^8) split into three
//         fp16 terms; the accumulators ARE the scores, no per-score FFMA / shared load.  For the bias to fit fp16 the
//         operands are scaled to 2^7..2^8 (not 2^13..2^14 as in K1; hi + lo still carry 22 bits);
//       - argmax AND a bound on every other score without packing indices: the 256 scores are a 16 x 16 matrix
//         (k = 16 g + j); R_g = max over row g and C_j = max over column j cost one FMNMX3 per two scores each.  The
//         best score is max R = max C at (g*, j*); every other candidate sits in another row or another column, so
//         max(second largest R, second largest C) bounds them all.  If best - that bound exceeds the error bound of the
//         prefilter (+ the fp32 direct form's own rounding) the pair is decided, else (row, sub-vector) goes to a pair
//         list and the fp32 direct-form arbiter (pq_fix_pairs_kernel) re-decides it in pq_encode_kernel's arithmetic;
//       - one thread owns all 256 scores of its (row, sub-vector): two epilogue groups (4 warps each) take alternate
//         sub-vectors, four 64-column tcgen05.ld each; a buffer goes back to the MMA warps as soon as it is in registers.
//
// Warps: 0 TMA producer ([128 rows x 32 fp32] boxes, 128B swizzle, 4 stages) | 1-2 MMA | 3 codebook-group loader |
// 4-7 converters (thread = row = TMEM lane; fp32 -> fp16 hi|lo into one of 3 TMEM operand stages; |x_j|^2 on the side) |
// 8-11, 12-15 epilogue groups.  TMEM: [0,384) three accumulator buffers, [384,480) operand stages, [480,496) constant tile.
// Barriers that several roles wait on in turn (accumulator full / empty) exist once per waiter: a parity wait is only
// sound when the same thread observes every phase of its barrier in order.
#pragma once

namespace pq256 {

constexpr int TMQ = 128, KQ = 256, DSQ = 32, GSQ = 3;  // DSQ: K extent of a sub-vector's contraction (widths 24 and 32 both use 32)
constexpr int NSXQ = 4, NSAQ = 3, NORMQ = 16, NACCQ = 3;
constexpr int X_STAGEQ = TMQ * DSQ * 4;       // 16 KB (12 KB used at sub-vector width 24)
constexpr int B_BLOCKQ = KQ * DSQ * 2;        // 16 KB: 256 rows x 64 B
constexpr int B_SUBQ = 3 * B_BLOCKQ;          // 48 KB: [hi][lo][bias: -|c|^2 / 2^8 in three fp16 terms, K slots 0-2]
constexpr int THREADSQ = 512;
constexpr int CONVQ_WARP0 = 4, CONVQ_WARPS = 4, EPIQ_WARP0 = 8, EPIQ_WARPS = 8;
constexpr uint32_t AQ_COL0 = 384, AQ_CONST = 480;
constexpr int SCALE_EXPQ = 7;                 // operands scaled to [2^7, 2^8)
constexpr float BIAS_A = 256.f;               // the constant operand of the bias MMA
// rounding of the fp32 direct form sum_e (x_e - c_e)^2 with four chains of 8 FMAs + 2 adds: <= 12 * 2^-24 of the sum,
// doubled for margin
constexpr float GAMMA_DIRECT = 12.f * 1.1920929e-7f;

struct PqParams {
  const float* X; int64_t n; int d; int M; int metric;
  const __half* Bimg;      // [M][3][KQ][DSQ] fp16, pre-swizzled
  const float* subc;       // [M][4]: e1max, B, cmax, unused
  const float* consts;
  int32_t* codes;          // [n][M]
  uint32_t* pairs; unsigned long long* pair_count; unsigned long long pair_cap; int* overflow;
  int* err_flag;
  int64_t n_tiles;
};

struct SmemQ {
  int x_off, b_off, subc_off, norm_off, bar_off, holder_off, total;
};
__host__ __device__ inline SmemQ smemq_layout() {
  SmemQ L;
  L.x_off = 0;
  L.b_off = L.x_off + NSXQ * X_STAGEQ;
  L.subc_off = L.b_off + GSQ * B_SUBQ;
  L.norm_off = L.subc_off + 64;
  L.bar_off = L.norm_off + NORMQ * TMQ * 4;
  L.holder_off = L.bar_off + 64 * 8;
  L.total = L.holder_off + 16;
  return L;
}

__device__ __forceinline__ float fmax3(float a, float b, float c) {
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}

// 64 scores (one 64-column load = matrix rows 4 i0 .. 4 i0 + 3) into the row maxima R and the column maxima C;
// i0 is a constant after unrolling, so R stays in registers
__device__ __forceinline__ void reduce64(const uint32_t (&ra)[64], const int i0, float (&R)[16], float (&C)[16]) {
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const uint32_t* v = ra + 16 * r;
    float m = fmax3(__uint_as_float(v[0]), __uint_as_float(v[1]), __uint_as_float(v[2]));
#pragma unroll
    for (int i = 3; i < 15; i += 2) m = fmax3(m, __uint_as_float(v[i]), __uint_as_float(v[i + 1]));
    R[4 * i0 + r] = fmaxf(m, __uint_as_float(v[15]));
  }
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    C[j] = fmax3(C[j], __uint_as_float(ra[j]), __uint_as_float(ra[16 + j]));
    C[j] = fmax3(C[j], __uint_as_float(ra[32 + j]), __uint_as_float(ra[48 + j]));
  }
}

// DS = sub-vector width: 32 (128-byte box rows, 128B swizzle) or 24 (96-byte box rows, no swizzle; K elements 24-31 are zero)
template <int DS>
__global__ void __launch_bounds__(THREADSQ, 1) pq_tensor_kernel(PqParams p, const __grid_constant__ CUtensorMap tmap) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const SmemQ L = smemq_layout();
  uint8_t* sX = smem + L.x_off;
  uint8_t* sB = smem + L.b_off;
  float* sSubc = reinterpret_cast<float*>(smem + L.subc_off);
  float* sNorm = reinterpret_cast<float*>(smem + L.norm_off);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.bar_off);
  uint64_t* x_full = bars;
  uint64_t* x_empty = x_full + NSXQ;
  uint64_t* a_full = x_empty + NSXQ;
  uint64_t* a_empty = a_full + NSAQ;
  uint64_t* st_full = a_empty + NSAQ;
  uint64_t* acc_full = st_full + NORMQ;         // [2 * buffer + epilogue group]
  uint64_t* acc_empty = acc_full + 2 * NACCQ;   // [2 * buffer + MMA warp that issues the buffer's next tenant]
  uint64_t* b_full = acc_empty + 2 * NACCQ;
  uint64_t* b_free = b_full + 1;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(smem + L.holder_off);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int M = p.M;
  const int ngroups = (M + GSQ - 1) / GSQ;

  if (warp == 1 && lane == 0) {
    for (int s = 0; s < NSXQ; ++s) { ptx::mbar_init(&x_full[s], 1); ptx::mbar_init(&x_empty[s], CONVQ_WARPS); }
    for (int s = 0; s < NSAQ; ++s) { ptx::mbar_init(&a_full[s], CONVQ_WARPS); ptx::mbar_init(&a_empty[s], 2); }
    for (int s = 0; s < NORMQ; ++s) ptx::mbar_init(&st_full[s], CONVQ_WARPS);
    for (int b = 0; b < 2 * NACCQ; ++b) { ptx::mbar_init(&acc_full[b], 1); ptx::mbar_init(&acc_empty[b], EPIQ_WARPS / 2); }
    ptx::mbar_init(b_full, 1);
    ptx::mbar_init(b_free, 2 + EPIQ_WARPS);
    ptx::mbar_fence_init();
  }
  if (warp == 0 && lane == 0) ptx::tma_prefetch_desc(&tmap);
  if (warp == 2) ptx::tmem_alloc(tmem_holder, TMEM_COLS);
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_holder;

  if (warp == 0) {
    // ===== TMA producer: one [128 x 32] fp32 box per (group, tile, sub-vector) =====
    uint32_t s = 0, ph = 0;
    for (int g = 0; g < ngroups; ++g) {
      const int gs = M - g * GSQ < GSQ ? M - g * GSQ : GSQ;
      for (int64_t tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
        for (int sv = 0; sv < gs; ++sv) {
          if (!__all_sync(MEVI_FULL_MASK, ptx::mbar_wait_backoff(&x_empty[s], ph ^ 1, 32))) {
            if (lane == 0) atomicExch(p.err_flag, 1);
            return;
          }
          if (ptx::elect_one()) {
            ptx::mbar_arrive_expect_tx(&x_full[s], TMQ * DS * 4);
            ptx::tma_load_2d(sX + (size_t)s * X_STAGEQ, &tmap, (g * GSQ + sv) * DS, (int)(tile * TMQ), &x_full[s]);
          }
          __syncwarp();
          if (++s == NSXQ) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 3) {
    // ===== codebook-group loader: images (hi | lo | bias) and bound constants of the group's sub-vectors =====
    for (int g = 0; g < ngroups; ++g) {
      const int gs = M - g * GSQ < GSQ ? M - g * GSQ : GSQ;
      if (g > 0 && !__all_sync(MEVI_FULL_MASK, ptx::mbar_wait_backoff(b_free, (g - 1) & 1, 64))) {
        if (lane == 0) atomicExch(p.err_flag, 7);
        return;
      }
      if (ptx::elect_one()) {
        ptx::mbar_arrive_expect_tx(b_full, (uint32_t)gs * (B_SUBQ + 16));
        const uint8_t* src = reinterpret_cast<const uint8_t*>(p.Bimg) + (size_t)g * GSQ * B_SUBQ;
        for (int i = 0; i < gs * (B_SUBQ / 16384); ++i) ptx::bulk_g2s(sB + (size_t)i * 16384, src + (size_t)i * 16384, 16384, b_full);
        ptx::bulk_g2s(sSubc, p.subc + (size_t)g * GSQ * 4, (uint32_t)gs * 16, b_full);
      }
      __syncwarp();
    }
  } else if (warp == 1 || warp == 2) {
    // ===== MMA: warp h issues the units (sub-vector, half h); unit u = 2q + h lives in accumulator buffer u % 3 =====
    const int h = warp - 1;
    const uint32_t idesc = ptx::umma_idesc_f16_m128(128u);
    uint32_t as = 0, aph = 0, q = 0, buf = (uint32_t)h, ebits = 0;
    for (int g = 0; g < ngroups; ++g) {
      const int gs = M - g * GSQ < GSQ ? M - g * GSQ : GSQ;
      if (!__all_sync(MEVI_FULL_MASK, ptx::mbar_wait_backoff(b_full, g & 1, 32))) {
        if (lane == 0) atomicExch(p.err_flag, 3);
        return;
      }
      for (int64_t tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
        const bool last_tile = tile + gridDim.x >= p.n_tiles;
        for (int sv = 0; sv < gs; ++sv, ++q) {
          // the buffer's previous tenant (unit u - 3, issued by the other MMA warp) must be drained
          if (2 * q + h >= NACCQ) {
            if (!__all_sync(MEVI_FULL_MASK, ptx::mbar_wait(&acc_empty[2 * buf + h], (ebits >> buf) & 1u))) {
              if (lane == 0) atomicExch(p.err_flag, 2);
              return;
            }
            ebits ^= 1u << buf;
          }
          const uint32_t d_tmem = tmem_base + buf * 128u;
          if (!__all_sync(MEVI_FULL_MASK, ptx::mbar_wait(&a_full[as], aph))) {
            if (lane == 0) atomicExch(p.err_flag, 3);
            return;
          }
          ptx::tc_fence_after_sync();
          const uint32_t b_hi = ptx::smem_u32(sB + (size_t)sv * B_SUBQ) + (uint32_t)h * 128u * 64u;
          const uint32_t b_lo = b_hi + (uint32_t)B_BLOCKQ, b_bias = b_lo + (uint32_t)B_BLOCKQ;
          if (ptx::elect_one()) {
            const uint32_t a_hi = tmem_base + AQ_COL0 + as * 32, a_lo = a_hi + 16;
            // scores = -|c_k|^2 (constant tile x bias block) + 2 x.c (the scales carry the factor): 7 MMAs
            ptx::umma_f16_ts(d_tmem, tmem_base + AQ_CONST, ptx::umma_desc_sw64(b_bias), idesc, 0u);
#pragma unroll
            for (int ks = 0; ks < DSQ / 16; ++ks) {
              ptx::umma_f16_ts(d_tmem, a_hi + ks * 8, ptx::umma_desc_sw64(b_hi + ks * 32), idesc, 1u);
              ptx::umma_f16_ts(d_tmem, a_hi + ks * 8, ptx::umma_desc_sw64(b_lo + ks * 32), idesc, 1u);
              ptx::umma_f16_ts(d_tmem, a_lo + ks * 8, ptx::umma_desc_sw64(b_hi + ks * 32), idesc, 1u);
            }
            ptx::umma_commit(&a_empty[as]);
            ptx::umma_commit(&acc_full[2 * buf + (q & 1)]);
            if (last_tile && sv == gs - 1) ptx::umma_commit(b_free);
          }
          __syncwarp();
          if (++as == NSAQ) { as = 0; aph ^= 1; }
          buf = buf >= 1 ? buf - 1 : buf + 2;  // (u + 2) % 3
        }
      }
    }
  } else if (warp >= CONVQ_WARP0 && warp < EPIQ_WARP0) {
    // ===== converters: thread = row; fp32 -> (hi | lo) fp16 into a TMEM operand stage, |x_j|^2 into the norm ring =====
    const int cw = warp - CONVQ_WARP0;
    const int row = cw * 32 + lane;
    const float sx = p.consts[C_SX], inv_sx2 = p.consts[C_INV_SX2];
    const float2 sx2 = make_float2(sx, sx);
    const uint32_t src_row = ptx::smem_u32(sX) + (uint32_t)row * (uint32_t)(DS * 4);
    const uint32_t sw = DS == 32 ? (uint32_t)(row & 7) : 0u;
    const uint32_t t_lane = tmem_base + ((uint32_t)(cw * 32) << 16);
    {  // the constant operand tile of the bias MMA: K slots 0-2 = 2^8, the rest 0 (the first publish below waits for it too)
      uint32_t ct[16];
      const __half2 aa = __floats2half2_rn(BIAS_A, BIAS_A), a0 = __floats2half2_rn(BIAS_A, 0.f);
      ct[0] = *reinterpret_cast<const uint32_t*>(&aa);
      ct[1] = *reinterpret_cast<const uint32_t*>(&a0);
#pragma unroll
      for (int i = 2; i < 16; ++i) ct[i] = 0u;
      ptx::tmem_st16(t_lane + AQ_CONST, ct);  // columns 480-495 (only 480-487 are read)
    }
    uint32_t xs = 0, xph = 0, as = 0, aph = 0, q = 0;
    for (int g = 0; g < ngroups; ++g) {
      const int gs = M - g * GSQ < GSQ ? M - g * GSQ : GSQ;
      for (int64_t tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
        for (int sv = 0; sv < gs; ++sv, ++q) {
          if (!ptx::mbar_wait(&x_full[xs], xph)) { atomicExch(p.err_flag, 4); return; }
          if (!ptx::mbar_wait_backoff(&a_empty[as], aph ^ 1, 32)) { atomicExch(p.err_flag, 4); return; }
          ptx::tc_fence_after_sync();
          uint32_t hi[16], lo[16];
          float2 norm2 = make_float2(0.f, 0.f);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float2 p01, p23;
            if (4 * j >= DS) {  // K padding of the narrow sub-vector
              hi[2 * j] = hi[2 * j + 1] = lo[2 * j] = lo[2 * j + 1] = 0u;
              continue;
            }
            asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(p01.x), "=f"(p01.y), "=f"(p23.x), "=f"(p23.y)
                         : "r"(src_row + xs * X_STAGEQ + (((uint32_t)j ^ sw) << 4)));
            p01 = ptx::f2_mul(p01, sx2);
            p23 = ptx::f2_mul(p23, sx2);
            norm2 = ptx::f2_fma(p01, p01, norm2);
            norm2 = ptx::f2_fma(p23, p23, norm2);
            const __half2 h01 = __float22half2_rn(p01), h23 = __float22half2_rn(p23);
            const __half2 l01 = __float22half2_rn(ptx::f2_sub(p01, __half22float2(h01)));
            const __half2 l23 = __float22half2_rn(ptx::f2_sub(p23, __half22float2(h23)));
            hi[2 * j] = *reinterpret_cast<const uint32_t*>(&h01);
            hi[2 * j + 1] = *reinterpret_cast<const uint32_t*>(&h23);
            lo[2 * j] = *reinterpret_cast<const uint32_t*>(&l01);
            lo[2 * j + 1] = *reinterpret_cast<const uint32_t*>(&l23);
          }
          ptx::tmem_st16(t_lane + AQ_COL0 + as * 32, hi);
          ptx::tmem_st16(t_lane + AQ_COL0 + as * 32 + 16, lo);
          sNorm[(q & (NORMQ - 1)) * TMQ + row] = (norm2.x + norm2.y) * inv_sx2;
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&x_empty[xs]);
          // publish at once: with three operand stages a publish delayed by one conversion (K1 hides the tcgen05.st
          // latency that way) would leave only two stages of overlap between conversion and MMA
          ptx::tmem_st_wait();
          ptx::tc_fence_before_sync();
          __syncwarp();
          if (lane == 0) { ptx::mbar_arrive(&a_full[as]); ptx::mbar_arrive(&st_full[q & (NORMQ - 1)]); }
          if (++xs == NSXQ) { xs = 0; xph ^= 1; }
          if (++as == NSAQ) { as = 0; aph ^= 1; }
        }
      }
    }
  } else {
    // ===== epilogue: group e takes the sub-vectors with (q & 1) == e; thread = (row, sub-vector), all 256 scores =====
    const int ew = warp - EPIQ_WARP0;
    const int e = ew >> 2, qd = ew & 3;
    const int rl = qd * 32 + lane;
    // score units -> accumulator units (acc = sx sc / f * s): the decision threshold is applied to raw accumulators
    const float to_acc = p.consts[C_SX] * p.consts[C_SC] * (p.metric == MEVI_METRIC_L2 ? 0.5f : 1.f);
    // |x_j|^2 below this guarantees that no scaled element overflowed the fp16 range
    const float xn2_limit = 65000.f * 65000.f * p.consts[C_INV_SX2];
    const uint32_t taddr = tmem_base + ((uint32_t)(qd * 32) << 16);
    uint32_t q = 0, fbits = 0;
    bool ok = true;
    for (int g = 0; g < ngroups && ok; ++g) {
      const int gs = M - g * GSQ < GSQ ? M - g * GSQ : GSQ;
      if (!ptx::mbar_wait_backoff(b_full, g & 1, 64)) { atomicExch(p.err_flag, 6); ok = false; break; }
      for (int64_t tile = blockIdx.x; tile < p.n_tiles && ok; tile += gridDim.x) {
        const int64_t row = tile * TMQ + rl;
        // a warp whose rows all lie past the end has nothing to reduce.  The branch also keeps ptxas from hoisting the
        // second tcgen05.ld above the first reduction: two live 64-score sets do not fit 128 registers and spill.
        const bool live = __any_sync(MEVI_FULL_MASK, row < p.n);
        for (int sv = 0; sv < gs; ++sv, ++q) {
          if ((int)(q & 1) != e) continue;
          // scores as a 16 x 16 matrix (k = 16 g + j): row maxima R[g], column maxima C[j]
          float R[16], C[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) { R[i] = -CUDART_INF_F; C[i] = -CUDART_INF_F; }
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const uint32_t buf = (2 * q + h) % NACCQ;
            if (!ptx::mbar_wait_backoff(&acc_full[2 * buf + e], (fbits >> buf) & 1u, 20)) { atomicExch(p.err_flag, 6); ok = false; break; }
            fbits ^= 1u << buf;
            ptx::tc_fence_after_sync();
            uint32_t ra[64];
            ptx::tmem_ld64(taddr + buf * 128u, ra);
            ptx::tmem_ld_wait();
            if (live) reduce64(ra, 2 * h, R, C);
            ptx::tmem_ld64(taddr + buf * 128u + 64u, ra);
            ptx::tmem_ld_wait();
            // the unit is in registers: hand the buffer to its next tenant (unit u + 3, the other half's MMA warp)
            ptx::tc_fence_before_sync();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(&acc_empty[2 * buf + (h ^ 1)]);
            if (live) reduce64(ra, 2 * h + 1, R, C);
          }
          if (!ok) break;
          if (!ptx::mbar_wait_backoff(&st_full[q & (NORMQ - 1)], (q >> 4) & 1, 32)) { atomicExch(p.err_flag, 6); ok = false; break; }
          const float xn2 = sNorm[(q & (NORMQ - 1)) * TMQ + rl];
          // largest and second largest (equal values count twice) of the row maxima and of the column maxima
          // (measured: running scans beat shallow compare / select trees here - fewer instructions on the ALU pipe)
          float r1 = -CUDART_INF_F, r2 = -CUDART_INF_F, c1 = -CUDART_INF_F, c2 = -CUDART_INF_F;
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            r2 = fmaxf(r2, fminf(r1, R[i]));
            r1 = fmaxf(r1, R[i]);
            c2 = fmaxf(c2, fminf(c1, C[i]));
            c1 = fmaxf(c1, C[i]);
          }
          int gi = 0, ji = 0;
#pragma unroll
          for (int i = 15; i >= 0; --i) {
            if (R[i] == r1) gi = i;
            if (C[i] == r1) ji = i;
          }
          const float xn = sqrtf(xn2);
          const float e1max = sSubc[sv * 4], bj = sSubc[sv * 4 + 1], cmax = sSubc[sv * 4 + 2];
          const float thr = (fmaf(2.f * xn, e1max, bj) + 2.f * GAMMA_DIRECT * (xn + cmax) * (xn + cmax)) * to_acc;
          const bool decided = (r1 - fmaxf(r2, c2) > thr) && (xn2 < xn2_limit) && (c1 == r1);
          const bool valid = row < p.n;
          const int m = g * GSQ + sv;
          if (valid) p.codes[row * M + m] = gi * 16 + ji;
          const bool flag = valid && !decided;
          const unsigned fm = __ballot_sync(MEVI_FULL_MASK, flag);
          if (fm != 0u) {
            const int leader = __ffs(fm) - 1;
            unsigned long long base = 0;
            if (lane == leader) base = atomicAdd(p.pair_count, (unsigned long long)__popc(fm));
            base = __shfl_sync(MEVI_FULL_MASK, base, leader);
            if (flag) {
              const unsigned long long slot = base + __popc(fm & ((1u << lane) - 1u));
              if (slot < p.pair_cap) p.pairs[slot] = (uint32_t)(row * M + m);
              else atomicExch(p.overflow, 1);
            }
          }
        }
      }
      // the group's images and constants may be overwritten once every epilogue warp (and both MMA warps) are done
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(b_free);
    }
  }

  ptx::tc_fence_before_sync();
  __syncthreads();
  if (warp == 2) ptx::tmem_dealloc(tmem_base, TMEM_COLS);
}

// scales for this kernel: 2^s with amax * 2^s in [2^7, 2^8) (the bias -|c|^2 sx sc / f / 2^8 must fit fp16)
__global__ void pq_scale_kernel(const unsigned* absmax2, int ds, float* consts) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    const float ac = __uint_as_float(absmax2[0]), ax = __uint_as_float(absmax2[1]);
    const float sc = ac > 0.f ? ldexpf(1.f, SCALE_EXPQ - ilogbf(ac)) : 1.f;
    float sx = ax > 0.f ? ldexpf(1.f, SCALE_EXPQ - ilogbf(ax)) : 1.f;
    // the bias |c|^2 sx sc / 512 <= 32 ac^2 sx sc / 512 < 2^4 ac sx must stay inside fp16: sx < 2^11 / ac (only binds when
    // the rows are much smaller than the centroids; their fp16 images then sit lower in the normal range, still 22 bits)
    if (ac > 0.f) sx = fminf(sx, ldexpf(1.f, 10 - ilogbf(ac)));
    consts[C_SC] = sc;
    consts[C_SX] = sx;
    consts[C_INV] = 1.f / (sc * sx);
    consts[C_INV_SX2] = (1.f / sx) * (1.f / sx);
    const float floor_abs = sqrtf((float)ds) * 5.9604645e-8f;  // sqrt(d) * 2^-24: fp16 subnormal spacing of hi+lo
    consts[C_FX] = floor_abs / sx;
    consts[C_FC] = floor_abs / sc;
  }
}

// Bimg[j][block][row][32 halfs], blocks hi(c*sc) | lo | bias; 16-byte units XOR-swizzled by (row>>1)&3 (UMMA 64B swizzle).
// bias row k: K slots 0-2 = three fp16 terms of  t_k / 2^8,  t_k = -|c_k|^2 sx sc / f  ('l2'; 0 for 'ip'), the rest 0.
__global__ void pq_bimg_kernel(const float* __restrict__ cb, int M, int ds, int metric, const float* __restrict__ consts,
                               __half* __restrict__ Bimg) {
  const int total = M * KQ * (DSQ / 8);
  const float sc = consts[C_SC], sx = consts[C_SX];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int u = i & 3, r = (i >> 2) & (KQ - 1), j = i >> 10;
    const float* crow = cb + ((size_t)j * KQ + r) * ds;
    __half hi[8], lo[8], bias[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float t = u * 8 + e < ds ? crow[u * 8 + e] * sc : 0.f;
      hi[e] = __float2half_rn(t);
      lo[e] = __float2half_rn(t - __half2float(hi[e]));
      bias[e] = __float2half_rn(0.f);
    }
    if (u == 0 && metric == MEVI_METRIC_L2) {
      double s = 0.0;
      for (int e = 0; e < ds; ++e) s += (double)crow[e] * (double)crow[e];
      // the fp32 value the bound constants assume, moved to accumulator units by exact power-of-two factors
      const float t = -(float)s * sx * sc * 0.5f * (1.f / BIAS_A);
      bias[0] = __float2half_rn(t);
      const float t1 = t - __half2float(bias[0]);
      bias[1] = __float2half_rn(t1);
      bias[2] = __float2half_rn(t1 - __half2float(bias[1]));
    }
    const int up = u ^ ((r >> 1) & 3);
    __half* base = Bimg + (size_t)j * (3 * KQ * DSQ);
    *reinterpret_cast<uint4*>(base + (size_t)r * DSQ + up * 8) = *reinterpret_cast<const uint4*>(hi);
    *reinterpret_cast<uint4*>(base + (size_t)(KQ + r) * DSQ + up * 8) = *reinterpret_cast<const uint4*>(lo);
    *reinterpret_cast<uint4*>(base + (size_t)(2 * KQ + r) * DSQ + up * 8) = *reinterpret_cast<const uint4*>(bias);
  }
}

// per sub-vector (one block of 256 threads, thread = centroid): the constants of the error bound
//   |score_k - exact| <= |x_j| * E1_k + B_j/2   (rq_tensor.cu, level_consts_kernel, with no Gram terms)
__global__ void pq_consts_kernel(const float* __restrict__ cb, int ds, int metric, const float* __restrict__ consts,
                                 float* __restrict__ subc) {
  const int j = blockIdx.x, k = threadIdx.x;
  const float f = metric == MEVI_METRIC_L2 ? 2.f : 1.f;
  const float EPS_A = 4.8e-7f;
  double s = 0.0;
  for (int e = 0; e < ds; ++e) {
    const double v = cb[((size_t)j * KQ + k) * ds + e];
    s += v * v;
  }
  const float c2 = (float)s, cn = (float)sqrt(s) * (1.f + 1e-6f);
  __shared__ float red[2][KQ / 32];
  float cmax = cn, c2max = c2;
  for (int o = 16; o > 0; o >>= 1) {
    cmax = fmaxf(cmax, __shfl_xor_sync(MEVI_FULL_MASK, cmax, o));
    c2max = fmaxf(c2max, __shfl_xor_sync(MEVI_FULL_MASK, c2max, o));
  }
  if ((k & 31) == 0) { red[0][k >> 5] = cmax; red[1][k >> 5] = c2max; }
  __syncthreads();
  if (k == 0) {
    for (int w = 1; w < KQ / 32; ++w) { cmax = fmaxf(cmax, red[0][w]); c2max = fmaxf(c2max, red[1][w]); }
    subc[j * 4 + 0] = f * (U_REL + EPS_A) * cmax + f * consts[C_FC];
    subc[j * 4 + 1] = 2.f * (f * consts[C_FX] * cmax + EPS_A * c2max);
    subc[j * 4 + 2] = cmax;
    subc[j * 4 + 3] = 0.f;
  }
}

}  // namespace pq256
