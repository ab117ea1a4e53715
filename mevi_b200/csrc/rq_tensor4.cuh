// rq_tensor4.cuh — K1, split-fp16 kernel (generation 4): the document operand goes through TENSOR MEMORY.
// The shipped K1 kernel for every supported shape (M = 1 - the k-means assignment - runs at the HBM roofline here).
//
// Same algorithm / error model / work-list protocol as the earlier generations (rq_tensor.cu).  v3 is bound
// by shared-memory bandwidth (70 % of the LSU data pipe: TMA writes + converter loads + converter stores +
// UMMA operand fetches = 19.5 KB per document).  Here the converters write the fp16 hi|lo operand tiles
// straight into TMEM with tcgen05.st and tcgen05.mma reads A from TMEM, which removes the converter stores
// and the A-operand fetches from shared memory (12 KB per document) and frees 64 KB of it for a deeper
// TMA ring:
//   warp 0      TMA producer: [256 rows x 32 fp32] boxes, 128B-swizzled, into a 4-stage ring (128 KB in flight)
//   warp 3      codebook producer: 16 KB bulk copies of the pre-swizzled [C_hi|C_lo] chunk image (4 stages, in lockstep with the operand stages)
//   warps 4-11  converters, ONE THREAD PER ROW (thread = TMEM lane): 8 conflict-free 16-byte loads of the row's
//               chunk, scale/split, 2 x tcgen05.st.x16 into one of 4 TMEM operand stages; the row norm is a
//               plain per-thread accumulator (no shuffles)
//   warps 1-2   tcgen05.mma with A in TMEM, one warp per 128-row half: per K step A_hi.C_hi + A_hi.C_lo + A_lo.C_hi
//               into the half's 128-column accumulator; ONE commit per warp and chunk releases operand + codebook stage
//   warps 12-19 epilogue, one row per thread (single accumulator buffer; the 4 TMEM operand stages keep the
//               converters busy while it drains)
// TMEM map (512 columns): [0,256) accumulators (half h at 128h), [256,512) 4 operand stages x (2 halves x (16 hi + 16 lo)).
#pragma once

namespace v4 {

constexpr int TM4 = 256;
constexpr int KC4 = 32;
constexpr int NSX4 = 4, NSB4 = 4, NSA4 = 4;
// Fused k-means variant (template argument ACC): the same pass also accumulates the per-centroid sums|counts of the
// rows under their PREVIOUS assignment (known before the pass), straight from the fp32 TMA stages:
//   warps 12-15  epilogue (4 warps instead of 8: each takes its TMEM lane quarter of both 128-row halves)
//   warp 16      sorter: per tile a stable counting sort of the 256 rows by previous code (bucket offsets + row list)
//                and the steps of the accumulation (every centroid's sorted rows cut into steps of 16)
//   warps 17-24  accumulators, per K chunk (32 columns) in two phases: A - the steps are dealt round-robin to the 8 warps
//                (balanced whatever the cluster sizes): 16 sorted rows per step, four independent 16-byte shared loads
//                per lane, partial sum parked in a staging buffer; B - warp a owns the centroids [K/8 * a, K/8 * (a+1))
//                and adds their steps' partials in step order to the CTA's [K][d] fp32 accumulators in shared memory.
//                No atomics, a fixed summation order: bit-reproducible.
// The accumulators take 96 KB of shared memory (K = 32, d = 768), so the fp32 ring is 3 stages deep instead of 4.
constexpr int NSX4_ACC = 3;
constexpr int EPI_WARPS4_ACC = 4;       // fused variant: the (light, single-level) epilogue runs on 4 warps, both halves each
constexpr int SORT_WARP = 16, ACC_WARP0 = 17, ACC_WARPS = 8;
constexpr int THREADS4_ACC = 32 * (ACC_WARP0 + ACC_WARPS);  // 800
constexpr int STEP_ROWS4 = 16;                       // sorted rows per accumulation step
constexpr int MAX_STEPS4 = TM4 / STEP_ROWS4 + 32;    // every centroid's list is cut into steps of 16 rows: <= 16 + K steps
static_assert(NSA4 == NSB4, "the A (TMEM) and B (smem) rings share their 'empty' barriers");
constexpr int X_STAGE4 = TM4 * KC4 * 4;  // 32 KB
constexpr int THREADS4 = 640;
constexpr int EPI_WARPS4 = 8;
constexpr uint32_t A_COL0 = 256;         // first TMEM column of the operand stages
struct Smem4 {
  int x_off, b_off, gram_off, cn2_off, e1_off, lvl_off, stats_off, bar_off, holder_off, acc_off, sort_off, total;
};
// acc_floats > 0: fused k-means variant (3-stage fp32 ring + [K][d] accumulators + sort buffers)
__host__ __device__ inline Smem4 smem4_layout(int M, int K, int NT, int acc_floats = 0) {
  Smem4 L;
  L.x_off = 0;
  L.b_off = L.x_off + (acc_floats > 0 ? NSX4_ACC : NSX4) * X_STAGE4;
  L.gram_off = L.b_off + NSB4 * (2 * NT) * 64;
  int gram_pad = 0;
  for (int j = 1; j < M; ++j) gram_pad += j * K * (K + 1);
  L.cn2_off = L.gram_off + gram_pad * 4;
  L.e1_off = L.cn2_off + NT * 4;
  L.lvl_off = L.e1_off + NT * 4;
  L.stats_off = L.lvl_off + 64;
  L.bar_off = (L.stats_off + 2 * TM4 * 4 + 7) & ~7;
  L.holder_off = L.bar_off + 40 * 8;
  L.acc_off = (L.holder_off + 16 + 127) & ~127;
  // sort buffers: [2 tile parities] x (row list 256 B + bucket offsets (K+2) ints), then K running counts
  L.sort_off = L.acc_off + acc_floats * 4;
  // + zero line (128 B), step tables [2] x (48 centroid bytes + 48 row-count bytes + (K+2) first-step ints), staging
  // [2][48][128 B], row table [2][48][16] bytes
  L.total = acc_floats > 0 ? ((L.sort_off + 2 * (TM4 + (K + 2) * 4) + 2 * K * 4 + 15) & ~15) + 128 +
                                 2 * (MAX_STEPS4 + MAX_STEPS4 + (K + 2) * 4) + 16 + 2 * MAX_STEPS4 * 128 +
                                 2 * MAX_STEPS4 * STEP_ROWS4
                           : L.holder_off + 16;
  return L;
}

template <bool SCALE, int NSX>
__device__ __forceinline__ void converter_loop4(const Params& p, uint8_t* sX, float* sStats, uint32_t tmem_base, uint64_t* x_full,
                                                uint64_t* x_empty, uint64_t* a_full, uint64_t* a_empty, uint64_t* st_full,
                                                int cw, int lane) {
  const int half = cw >> 2;                       // warps 4-7 -> rows 0..127, warps 8-11 -> rows 128..255
  const int rl = (cw & 3) * 32 + lane;            // row inside the half == TMEM lane
  const int row = half * 128 + rl;                // row inside the tile == row of the TMA box
  const float sx = p.consts[C_SX], inv_sx2 = p.consts[C_INV_SX2];
  const int nchunks = p.d / KC4;
  const uint32_t src_row = ptx::smem_u32(sX) + (uint32_t)row * 128u;
  const uint32_t sw = (uint32_t)(row & 7);        // 128B swizzle: 16-byte chunk j of this row sits at j ^ (row & 7)
  const uint32_t t_lane = tmem_base + ((uint32_t)((cw & 3) * 32) << 16) + A_COL0 + (uint32_t)half * 32u;
  float2 norm2 = make_float2(0.f, 0.f);  // (even, odd) partial sums of the squared row norm
  const float2 sx2 = make_float2(sx, sx);
  uint32_t xs = 0, xph = 0, as = 0, aph = 0, it = 0, pend_stage = 0;
  bool pending = false;
  for (int64_t tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++it) {
    for (int c = 0; c < nchunks; ++c) {
      if (!ptx::mbar_wait(&x_full[xs], xph)) { atomicExch(p.err_flag, 4); return; }
      if (!ptx::mbar_wait_backoff(&a_empty[as], aph ^ 1, 32)) { atomicExch(p.err_flag, 4); return; }
      ptx::tc_fence_after_sync();
      uint32_t hi[16], lo[16];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float2 p01, p23;
        asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(p01.x), "=f"(p01.y), "=f"(p23.x), "=f"(p23.y)
                     : "r"(src_row + xs * X_STAGE4 + (((uint32_t)j ^ sw) << 4)));
        // packed fp32 pairs (FMUL2 / FFMA2 / FADD2): a quarter fewer issue slots -- and joules -- per converted float
        if (SCALE) { p01 = ptx::f2_mul(p01, sx2); p23 = ptx::f2_mul(p23, sx2); }
        norm2 = ptx::f2_fma(p01, p01, norm2);
        norm2 = ptx::f2_fma(p23, p23, norm2);
        const __half2 h01 = __float22half2_rn(p01), h23 = __float22half2_rn(p23);
        const __half2 l01 = __float22half2_rn(ptx::f2_sub(p01, __half22float2(h01)));
        const __half2 l23 = __float22half2_rn(ptx::f2_sub(p23, __half22float2(h23)));
        hi[2 * j] = *reinterpret_cast<const uint32_t*>(&h01);       // K elements 4j, 4j+1
        hi[2 * j + 1] = *reinterpret_cast<const uint32_t*>(&h23);   // K elements 4j+2, 4j+3
        lo[2 * j] = *reinterpret_cast<const uint32_t*>(&l01);
        lo[2 * j + 1] = *reinterpret_cast<const uint32_t*>(&l23);
      }
      // publish the PREVIOUS chunk's operand stage: its tcgen05.st had this chunk's conversion time to land
      if (pending) {
        ptx::tmem_st_wait();
        ptx::tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&a_full[pend_stage]);
      }
      ptx::tmem_st16(t_lane + as * 64, hi);
      ptx::tmem_st16(t_lane + as * 64 + 16, lo);
      // the stores consumed every value loaded from the X stage: hand it back to the TMA producer
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&x_empty[xs]);
      pending = true;
      pend_stage = as;
      if (++xs == NSX) { xs = 0; xph ^= 1; }
      if (++as == NSA4) { as = 0; aph ^= 1; }
    }
    // end of tile: publish its last operand stage right away (the MMA needs it to finish the tile)
    if (pending) {
      ptx::tmem_st_wait();
      ptx::tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&a_full[pend_stage]);
      pending = false;
    }
    sStats[(it & 1) * TM4 + row] = SCALE ? (norm2.x + norm2.y) * inv_sx2 : norm2.x + norm2.y;
    norm2 = make_float2(0.f, 0.f);
    __syncwarp();
    if (lane == 0) ptx::mbar_arrive(&st_full[it & 1]);
  }
}

template <int M, bool ACC>
__global__ void __launch_bounds__(ACC ? THREADS4_ACC : THREADS4, 1)
rq_tensor4_kernel(Params p, const __grid_constant__ CUtensorMap tmap) {
  extern __shared__ __align__(1024) uint8_t smem[];
  static_assert(!ACC || M == 1, "the fused accumulation is the k-means (single level) form");
  constexpr int NSX = ACC ? NSX4_ACC : NSX4;
  constexpr int NTHREADS = ACC ? THREADS4_ACC : THREADS4;
  const int K = p.K, NT = p.NT;
  const Smem4 L = smem4_layout(M, K, NT, ACC ? K * p.d : 0);
  uint8_t* sX = smem + L.x_off;
  uint8_t* sB = smem + L.b_off;
  float* sGram = reinterpret_cast<float*>(smem + L.gram_off);
  float* sCn2 = reinterpret_cast<float*>(smem + L.cn2_off);
  float* sE1 = reinterpret_cast<float*>(smem + L.e1_off);
  float* sLvl = reinterpret_cast<float*>(smem + L.lvl_off);
  float* sStats = reinterpret_cast<float*>(smem + L.stats_off);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.bar_off);
  uint64_t* x_full = bars;
  uint64_t* x_empty = x_full + NSX;
  uint64_t* a_full = x_empty + NSX;
  uint64_t* a_empty = a_full + NSA4;
  uint64_t* b_full = a_empty + NSA4;
  uint64_t* b_empty = b_full + NSB4;
  uint64_t* acc_full = b_empty + NSB4;
  uint64_t* acc_empty = acc_full + 1;
  uint64_t* st_full = acc_empty + 1;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(smem + L.holder_off);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t b_stage_bytes = (uint32_t)(2 * NT) * 64u;
  const int nchunks = p.d / KC4;

  for (int i = tid; i < p.gram_floats; i += NTHREADS) {
    const int r = i / K, c = i - r * K;
    sGram[r * (K + 1) + c] = p.gram[i];
  }
  for (int i = tid; i < NT; i += NTHREADS) {
    sCn2[i] = p.cn2[i];
    sE1[i] = p.e1[i];
  }
  for (int i = tid; i < M * 4; i += NTHREADS) sLvl[i] = p.lvl[i];
  // fused k-means accumulation: CTA-wide [K][d] sums, per tile parity a row list + bucket offsets, running counts
  float* sAcc = reinterpret_cast<float*>(smem + L.acc_off);
  uint8_t* sPerm = smem + L.sort_off;                                                  // [2][TM4]
  int* sOff = reinterpret_cast<int*>(smem + L.sort_off + 2 * TM4);                     // [2][K + 2]
  int* sCnt = sOff + 2 * (K + 2);                                                      // [K] rows per centroid so far (CTA)
  int* sRun = sCnt + K;                                                                // [K] sorter scratch
  const uint32_t zero_line = (ptx::smem_u32(sRun + K) + 15u) & ~15u;                   // 128 zero bytes (a row that adds nothing)
  uint8_t* sTab = smem + (((L.sort_off + 2 * (TM4 + (K + 2) * 4) + 2 * K * 4 + 15) & ~15) + 128);
  uint8_t* sStepB = sTab;                                                              // [2][MAX_STEPS4] centroid of a step
  uint8_t* sStepC = sTab + 2 * MAX_STEPS4;                                             // [2][MAX_STEPS4] rows of a step (1..16)
  int* sStep0 = reinterpret_cast<int*>(sTab + 4 * MAX_STEPS4);                         // [2][K + 2] first step of a centroid; [K] = count
  float4* sPart = reinterpret_cast<float4*>(sTab + ((2 * (MAX_STEPS4 + MAX_STEPS4 + (K + 2) * 4) + 15) & ~15));  // [2][MAX_STEPS4][8]
  uint8_t* sRowIdx = reinterpret_cast<uint8_t*>(sPart) + 2 * MAX_STEPS4 * 128;         // [2][MAX_STEPS4][16] row (in the tile) of every step row
  uint64_t* sort_full = st_full + 2;                                                   // [2]
  uint64_t* sort_empty = sort_full + 2;                                                // [2]
  if (ACC) {
    for (int i = tid; i < K * p.d; i += NTHREADS) sAcc[i] = 0.f;
    for (int i = tid; i < K; i += NTHREADS) sCnt[i] = 0;
    if (tid < 32) asm volatile("st.shared.b32 [%0], %1;" ::"r"(zero_line + tid * 4), "r"(0) : "memory");
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < NSX; ++s) { ptx::mbar_init(&x_full[s], 1); ptx::mbar_init(&x_empty[s], CONV_WARPS + (ACC ? ACC_WARPS : 0)); }
    if (ACC) {
      for (int b = 0; b < 2; ++b) { ptx::mbar_init(&sort_full[b], 1); ptx::mbar_init(&sort_empty[b], ACC_WARPS); }
    }
    for (int s = 0; s < NSA4; ++s) { ptx::mbar_init(&a_full[s], CONV_WARPS); ptx::mbar_init(&a_empty[s], 2); }  // one commit per MMA warp
    for (int s = 0; s < NSB4; ++s) { ptx::mbar_init(&b_full[s], 1); ptx::mbar_init(&b_empty[s], 1); }
    ptx::mbar_init(acc_full, 2);
    ptx::mbar_init(acc_empty, ACC ? EPI_WARPS4_ACC : EPI_WARPS4);
    ptx::mbar_init(&st_full[0], CONV_WARPS);
    ptx::mbar_init(&st_full[1], CONV_WARPS);
    ptx::mbar_fence_init();
  }
  if (warp == 0 && lane == 0) ptx::tma_prefetch_desc(&tmap);
  if (warp == 2) ptx::tmem_alloc(tmem_holder, TMEM_COLS);
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_holder;

  // The three control warps walk their loops with all 32 lanes (operands stay warp-uniform) and issue from one
  // elected lane: `if (lane == 0)` would wrap every TMA / tcgen05 instruction in an R2UR waterfall loop.
  if (warp == 0) {
    uint32_t s = 0, ph = 0;
    for (int64_t tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
      for (int c = 0; c < nchunks; ++c) {
        if (!__all_sync(MEVI_FULL_MASK, ptx::mbar_wait_backoff(&x_empty[s], ph ^ 1, 32))) {
          if (lane == 0) atomicExch(p.err_flag, 1);
          return;
        }
        if (ptx::elect_one()) {
          ptx::mbar_arrive_expect_tx(&x_full[s], X_STAGE4);
          ptx::tma_load_2d(sX + (size_t)s * X_STAGE4, &tmap, c * KC4, (int)(tile * TM4), &x_full[s]);
        }
        __syncwarp();
        if (++s == NSX) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 3) {
    uint32_t s = 0, ph = 0;
    for (int64_t tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
      for (int c = 0; c < nchunks; ++c) {
        if (!__all_sync(MEVI_FULL_MASK, ptx::mbar_wait_backoff(&a_empty[s], ph ^ 1, 32))) {
          if (lane == 0) atomicExch(p.err_flag, 7);
          return;
        }
        if (ptx::elect_one()) {
          ptx::mbar_arrive_expect_tx(&b_full[s], b_stage_bytes);
          ptx::bulk_g2s(sB + (size_t)s * b_stage_bytes, p.Bimg + (size_t)c * (2 * NT) * KC4, b_stage_bytes, &b_full[s]);
        }
        __syncwarp();
        if (++s == NSB4) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1 || warp == 2) {
    // TWO MMA warps, one per 128-row half (own accumulator, own commits): a single issuing thread leaves a
    // bubble in the tensor pipe after every tcgen05.commit; two independent streams fill each other's bubbles
    // (tools/umma_rate.cu: 12 TS MMAs + 2 commits per chunk in ~850 cycles instead of ~1630).
    const int h = warp - 1;
    const uint32_t idesc = ptx::umma_idesc_f16_m128((uint32_t)NT);
    const uint32_t d_tmem = tmem_base + h * 128;
    uint32_t as = 0, aph = 0, it = 0;
    for (int64_t tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++it) {
      // single accumulator buffer: the previous tile's epilogue must have drained it
      if (!__all_sync(MEVI_FULL_MASK, ptx::mbar_wait(acc_empty, (it & 1) ^ 1))) {
        if (lane == 0) atomicExch(p.err_flag, 2);
        return;
      }
      ptx::tc_fence_after_sync();
      for (int c = 0; c < nchunks; ++c) {
        if (!__all_sync(MEVI_FULL_MASK, ptx::mbar_wait(&a_full[as], aph))) {
          if (lane == 0) atomicExch(p.err_flag, 3);
          return;
        }
        if (!__all_sync(MEVI_FULL_MASK, ptx::mbar_wait(&b_full[as], aph))) {
          if (lane == 0) atomicExch(p.err_flag, 3);
          return;
        }
        ptx::tc_fence_after_sync();
        const uint32_t b_hi = ptx::smem_u32(sB + (size_t)as * b_stage_bytes);
        const uint32_t b_lo = b_hi + (uint32_t)NT * 64u;
        if (ptx::elect_one()) {
          const uint32_t a_hi = tmem_base + A_COL0 + as * 64 + h * 32, a_lo = a_hi + 16;
#pragma unroll
          for (int ks = 0; ks < KC4 / 16; ++ks) {
            ptx::umma_f16_ts(d_tmem, a_hi + ks * 8, ptx::umma_desc_sw64(b_hi + ks * 32), idesc, (c | ks) != 0 ? 1u : 0u);
            ptx::umma_f16_ts(d_tmem, a_hi + ks * 8, ptx::umma_desc_sw64(b_lo + ks * 32), idesc, 1u);
            ptx::umma_f16_ts(d_tmem, a_lo + ks * 8, ptx::umma_desc_sw64(b_hi + ks * 32), idesc, 1u);
          }
          // the operand (TMEM) and codebook (smem) rings advance in lockstep: converters and the codebook producer
          // both wait on a_empty[as], which completes when BOTH MMA warps have committed
          ptx::umma_commit(&a_empty[as]);
          if (c == nchunks - 1) ptx::umma_commit(acc_full);
        }
        __syncwarp();
        if (++as == NSA4) { as = 0; aph ^= 1; }
      }
    }
  } else if (warp >= CONV_WARP0 && warp < EPI_WARP0) {
    if (p.consts[C_SX] == 1.f)
      converter_loop4<false, NSX>(p, sX, sStats, tmem_base, x_full, x_empty, a_full, a_empty, st_full, warp - CONV_WARP0, lane);
    else
      converter_loop4<true, NSX>(p, sX, sStats, tmem_base, x_full, x_empty, a_full, a_empty, st_full, warp - CONV_WARP0, lane);
  } else if (ACC && warp == SORT_WARP) {
    // ===== sorter: stable counting sort of the tile's rows by PREVIOUS code; rows past the end go to bucket K =====
    uint32_t it = 0;
    for (int64_t tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++it) {
      const uint32_t buf = it & 1, bph = (it >> 1) & 1;
      if (!__all_sync(MEVI_FULL_MASK, ptx::mbar_wait_backoff(&sort_empty[buf], bph ^ 1, 64))) {
        if (lane == 0) atomicExch(p.err_flag, 8);
        return;
      }
      int code[TM4 / 32];
#pragma unroll
      for (int i = 0; i < TM4 / 32; ++i) {
        const int64_t row = tile * TM4 + i * 32 + lane;
        int c = K;
        if (row < p.n) {
          c = p.prev[row * p.prev_stride];
          c = c < 0 ? 0 : (c >= K ? K - 1 : c);
        }
        code[i] = c;
      }
      int* off = sOff + buf * (K + 2);
      // 1. bucket sizes: the first lane of every group of equal codes adds the group's size (distinct codes, distinct words)
      if (lane <= K && lane < 32) off[lane] = 0;
      if (lane == 0) off[K] = 0;
      __syncwarp();
#pragma unroll
      for (int i = 0; i < TM4 / 32; ++i) {
        const unsigned same = __match_any_sync(MEVI_FULL_MASK, code[i]);
        if (lane == __ffs(same) - 1) off[code[i]] += __popc(same);
        __syncwarp();
      }
      // 2. exclusive scan over the K (<= 32) buckets, lane = bucket; running counts of the CTA; placement counters
      const int cnt = lane < K ? off[lane] : 0;
      int incl = cnt;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(MEVI_FULL_MASK, incl, o);
        if (lane >= o) incl += v;
      }
      const int total_valid = __shfl_sync(MEVI_FULL_MASK, incl, 31);
      __syncwarp();
      if (lane < K) {
        off[lane] = incl - cnt;
        sCnt[lane] += cnt;
        sRun[lane] = 0;
      }
      if (lane == 0) off[K] = total_valid;
      __syncwarp();
      // 3. placement, rows in ascending order inside a bucket (stable): position = bucket start + rows of the bucket
      //    placed by earlier blocks + rank among the equal codes of this block
#pragma unroll
      for (int i = 0; i < TM4 / 32; ++i) {
        const int c = code[i];
        const unsigned same = __match_any_sync(MEVI_FULL_MASK, c);
        if (c < K) sPerm[buf * TM4 + off[c] + sRun[c] + __popc(same & ((1u << lane) - 1u))] = (uint8_t)(i * 32 + lane);
        __syncwarp();
        if (c < K && lane == __ffs(same) - 1) sRun[c] += __popc(same);
        __syncwarp();
      }
      // 4. steps: centroid `lane`'s list is cut into ceil(cnt / 16) steps; steps are numbered centroid by centroid
      {
        const int nst = lane < K ? (cnt + STEP_ROWS4 - 1) / STEP_ROWS4 : 0;
        int sincl = nst;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int v = __shfl_up_sync(MEVI_FULL_MASK, sincl, o);
          if (lane >= o) sincl += v;
        }
        int* st0 = sStep0 + buf * (K + 2);
        if (lane < K) st0[lane] = sincl - nst;
        if (lane == 31) st0[K] = sincl;
        for (int t = 0; t < nst; ++t) {
          sStepB[buf * MAX_STEPS4 + sincl - nst + t] = (uint8_t)lane;
          sStepC[buf * MAX_STEPS4 + sincl - nst + t] = (uint8_t)(cnt - STEP_ROWS4 * t < STEP_ROWS4 ? cnt - STEP_ROWS4 * t : STEP_ROWS4);
        }
      }
      __syncwarp();
      // 5. per step the stage offsets of its 16 rows (two steps per pass: lane = (step parity, row of the step))
      {
        const int total_steps = sStep0[buf * (K + 2) + K];
        for (int s2 = 0; s2 < total_steps; s2 += 2) {
          const int st = s2 + (lane >> 4), t = lane & 15;
          if (st < total_steps) {
            const int b = sStepB[buf * MAX_STEPS4 + st];
            const int q = off[b] + STEP_ROWS4 * (st - sStep0[buf * (K + 2) + b]) + t;
            sRowIdx[(buf * MAX_STEPS4 + st) * STEP_ROWS4 + t] = q < off[b + 1] ? sPerm[buf * TM4 + q] : (uint8_t)0;
          }
        }
      }
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&sort_full[buf]);
    }
  } else if (ACC && warp >= ACC_WARP0) {
    // ===== accumulators: sums of the rows under their previous code, from the fp32 stages =====
    const int aw = warp - ACC_WARP0;
    const int kb0 = aw * (K / ACC_WARPS), kb1 = (aw + 1) * (K / ACC_WARPS);
    const int d = p.d;
    const int g4 = lane >> 3;
    const uint32_t u8 = (uint32_t)(lane & 7);
    uint32_t xs = 0, xph = 0, it = 0;
    for (int64_t tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++it) {
      const uint32_t buf = it & 1, bph = (it >> 1) & 1;
      if (!ptx::mbar_wait_backoff(&sort_full[buf], bph, 64)) { atomicExch(p.err_flag, 9); return; }
      const uint8_t* perm = sPerm + buf * TM4;
      const int* off = sOff + buf * (K + 2);
      const uint8_t* stepb = sStepB + buf * MAX_STEPS4;
      const int* step0 = sStep0 + buf * (K + 2);
      const uint8_t* rowidx = sRowIdx + buf * MAX_STEPS4 * STEP_ROWS4;
      const uint8_t* stepc = sStepC + buf * MAX_STEPS4;
      for (int c = 0; c < nchunks; ++c) {
        if (!ptx::mbar_wait(&x_full[xs], xph)) { atomicExch(p.err_flag, 9); return; }
        // Phase A (balanced whatever the cluster sizes): the tile's steps are dealt to the 8 warps four at a time.  lane =
        // (step g = lane / 8 of the four, 16-byte unit u = lane % 8): one LDS.128 per lane covers one row of each of the
        // four steps x 32 columns per warp instruction.  A group of 8 lanes walks its step's (up to 16) sorted rows four
        // at a time (rows past the end read the zero line), adds them in a fixed order and parks the 32-column partial
        // sum in the staging buffer of this chunk's parity.
        const uint32_t stage_u32 = ptx::smem_u32(sX) + xs * X_STAGE4;
        float4* part = sPart + (c & 1) * MAX_STEPS4 * 8;
        const int nsteps = step0[K];
        for (int base = aw * 4; base < nsteps; base += 4 * ACC_WARPS) {
          // four steps per warp at a time, one per group of 8 lanes: no cross-lane reduction, 4 independent row streams.
          // The sorter left every step's 16 row offsets in a table (0xFFFF = past the end of the list -> zero line).
          const int sidx = base + g4;
          const bool live = sidx < nsteps;
          const uint8_t* ro = rowidx + (live ? sidx : 0) * STEP_ROWS4;
          const int cnt = live ? (int)stepc[sidx] : 0;
          float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0, a2 = a0, a3 = a0;
#pragma unroll
          for (int t0 = 0; t0 < STEP_ROWS4; t0 += 4) {
            if (__all_sync(MEVI_FULL_MASK, t0 >= cnt)) break;  // every group's list has ended
            const uint32_t r4 = *reinterpret_cast<const uint32_t*>(ro + t0);  // four row indices
            float4 v[4];
#pragma unroll
            for (int t = 0; t < 4; ++t) {
              const uint32_t r = (r4 >> (8 * t)) & 255u;
              const uint32_t ad = t0 + t < cnt ? stage_u32 + (r << 7) + ((u8 ^ (r & 7u)) << 4) : zero_line + (u8 << 4);
              asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v[t].x), "=f"(v[t].y), "=f"(v[t].z), "=f"(v[t].w) : "r"(ad));
            }
            a0.x += v[0].x; a0.y += v[0].y; a0.z += v[0].z; a0.w += v[0].w;
            a1.x += v[1].x; a1.y += v[1].y; a1.z += v[1].z; a1.w += v[1].w;
            a2.x += v[2].x; a2.y += v[2].y; a2.z += v[2].z; a2.w += v[2].w;
            a3.x += v[3].x; a3.y += v[3].y; a3.z += v[3].z; a3.w += v[3].w;
          }
          if (live)
            part[sidx * 8 + u8] = make_float4((a0.x + a1.x) + (a2.x + a3.x), (a0.y + a1.y) + (a2.y + a3.y),
                                              (a0.z + a1.z) + (a2.z + a3.z), (a0.w + a1.w) + (a2.w + a3.w));
        }
        // the fp32 stage is consumed: hand it back, then wait for every warp's partials (named barrier of the 8 warps)
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&x_empty[xs]);
        asm volatile("bar.sync 2, %0;" ::"n"(32 * ACC_WARPS) : "memory");
        // Phase B: warp a owns the centroids [K/8 * a, K/8 * (a+1)) and adds their steps' partials, in step order, to the
        // CTA's running sums (lanes 0-7: 32 columns).  The staging buffer of the other parity is free for the next
        // chunk's phase A: a warp passes the next barrier only after its own phase B.
        {  // lane = (g: which of the warp's K/8 centroids, u: 16-byte unit of the 32 columns)
          const int b = kb0 + g4;
          if (g4 < kb1 - kb0) {
            const int s0 = step0[b], s1 = step0[b + 1];
            if (s1 > s0) {
              float4 a = part[s0 * 8 + u8];
              for (int t = s0 + 1; t < s1; ++t) {
                const float4 w = part[t * 8 + u8];
                a.x += w.x; a.y += w.y; a.z += w.z; a.w += w.w;
              }
              float4* dst = reinterpret_cast<float4*>(sAcc + (size_t)b * d + c * KC4 + 4 * (int)u8);
              float4 t4 = *dst;
              t4.x += a.x; t4.y += a.y; t4.z += a.z; t4.w += a.w;
              *dst = t4;
            }
          }
        }
        if (++xs == NSX) { xs = 0; xph ^= 1; }
      }
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&sort_empty[buf]);
    }
  } else if (warp >= EPI_WARP0 && warp < EPI_WARP0 + (ACC ? EPI_WARPS4_ACC : EPI_WARPS4)) {
    const int ew = warp - EPI_WARP0;
    const float m2inv = (p.metric == MEVI_METRIC_L2 ? -2.f : -1.f) * p.consts[C_INV];
    const bool l2 = p.metric == MEVI_METRIC_L2;
    double inertia_acc = 0.0;
    uint32_t it = 0;
    bool ok = true;
    for (int64_t tile = blockIdx.x; tile < p.n_tiles && ok; tile += gridDim.x, ++it) {
      if (!ptx::mbar_wait_backoff(acc_full, it & 1, 64) || !ptx::mbar_wait_backoff(&st_full[it & 1], (it >> 1) & 1, 32)) { atomicExch(p.err_flag, 6); ok = false; break; }
      ptx::tc_fence_after_sync();
      // (fused k-means variant: 4 epilogue warps, each takes its lane quarter of BOTH halves)
      for (int h = ACC ? 0 : (ew >> 2); h < (ACC ? 2 : (ew >> 2) + 1); ++h) {
        const int q = ew & 3;  // 32-lane quarter of TMEM (== warp % 4)
        const int rl = h * 128 + q * 32 + lane;
        const float xn2 = sStats[(it & 1) * TM4 + rl];
        const float xn = sqrtf(xn2), nxn = -xn;
        const uint32_t taddr = tmem_base + h * 128 + ((uint32_t)(q * 32) << 16);
        const int64_t row = tile * TM4 + rl;
        int code[M];
        int flag_level = -1;
        float last_best = 0.f;
#pragma unroll
        for (int j = 0; j < M; ++j) code[j] = 0;
#pragma unroll
        for (int j = 0; j < M; ++j) {
          const float* gj = sGram + (j * (j - 1) / 2) * K * (K + 1);
          const float* grow[M > 1 ? M - 1 : 1];
#pragma unroll
          for (int m = 0; m < j; ++m) grow[m] = gj + (m * K + code[m]) * (K + 1);
          float m1 = CUDART_INF_F, ub = CUDART_INF_F, eb = 0.f, u1 = CUDART_INF_F, u2 = CUDART_INF_F;
          int besti = 0;
          for (int k0 = 0; k0 < K; k0 += 32) {
            uint32_t ra[32];
            ptx::tmem_ld32(taddr + j * K + k0, ra);
            ptx::tmem_ld_wait();
            float dk[32];
            float c1 = CUDART_INF_F;
#pragma unroll
            for (int kk = 0; kk < 32; ++kk) {
              float base = l2 ? sCn2[j * K + k0 + kk] : 0.f;
              float g = 0.f;
#pragma unroll
              for (int m = 0; m < j; ++m) g += grow[m][k0 + kk];
              base = l2 ? fmaf(2.f, g, base) : g;
              dk[kk] = fmaf(__uint_as_float(ra[kk]), m2inv, base);
              c1 = fminf(c1, dk[kk]);
              const float u = fmaf(nxn, sE1[j * K + k0 + kk], dk[kk]);
              u2 = fminf(u2, fmaxf(u1, u));
              u1 = fminf(u1, u);
            }
            int ci = 0;
#pragma unroll
            for (int kk = 31; kk >= 0; --kk)
              if (dk[kk] == c1) ci = kk;
            if (c1 < m1) {
              m1 = c1;
              besti = k0 + ci;
              eb = xn * sE1[j * K + besti];
              ub = fmaf(nxn, sE1[j * K + besti], c1);
            }
          }
          code[j] = besti;
          const float other_lo = (ub == u1) ? u2 : u1;
          const bool clear = other_lo > m1 + eb + sLvl[j * 4 + 1];
          if (!clear && flag_level < 0) flag_level = j;
          last_best = m1;
        }
        if (row < p.n) {
          int32_t* dst = p.codes + row * p.codes_stride;
          if (M == 4 && p.codes_stride == 4) {
            *reinterpret_cast<int4*>(dst) = make_int4(code[0], code[M > 1 ? 1 : 0], code[M > 2 ? 2 : 0], code[M > 3 ? 3 : 0]);
          } else {
#pragma unroll
            for (int j = 0; j < M; ++j) dst[j] = code[j];
          }
          if (flag_level >= 0) {
            const unsigned long long slot = atomicAdd(p.work_count, 1ull);
            p.work_rows[slot] = (int32_t)row;
            p.work_levels[slot] = flag_level;
          }
          if (p.inertia) inertia_acc += (double)(l2 ? fmaxf(last_best + xn2, 0.f) : -last_best);
        }
      }
      ptx::tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(acc_empty);
    }
    if (p.inertia) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) inertia_acc += __shfl_xor_sync(MEVI_FULL_MASK, inertia_acc, o);
      if (lane == 0 && inertia_acc != 0.0) atomicAdd(p.inertia, inertia_acc);
    }
  }

  ptx::tc_fence_before_sync();
  __syncthreads();
  if (warp == 2) ptx::tmem_dealloc(tmem_base, TMEM_COLS);
  if (ACC) {  // per-CTA partials; reduced in CTA order by kmeans_reduce_partials_kernel (deterministic)
    const int64_t kd = (int64_t)K * p.d;
    for (int i = tid; i < kd; i += NTHREADS) p.part_sums[(int64_t)blockIdx.x * kd + i] = sAcc[i];
    for (int i = tid; i < K; i += NTHREADS) p.part_counts[(int64_t)blockIdx.x * K + i] = sCnt[i];
  }
}

}  // namespace v4
