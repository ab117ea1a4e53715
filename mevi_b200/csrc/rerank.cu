// rerank.cu — K3 cluster-restricted re-rank (gather + dot + fused top-k) and K4 top-k merge.
//
// Replaces MEVI/main_models.py:3915-4014: for each query, walk its beam-search
// leaves in order, look the leaf up in the inverted lists (doc_cluster.get,
// 3928), gather the candidate rows (3944), score q.p (document_encoder.py:132)
// and sort descending (4012-4014) — here keeping only the k best.
//
// Data layout: inverted lists are CSR (leaf_offsets int64 [n_leaves+1],
// leaf_docids int32 [n]); a candidate is one 4*d-byte row of D, read exactly
// once per (query, candidate) with 128-bit loads, 512 contiguous bytes per warp
// instruction (a 3 KB row is 6 such instructions), so gathered rows are fully
// coalesced even though consecutive candidates are scattered.
// One CTA handles one (query, split) pair: the query's candidate range is cut
// into S equal splits so that small query batches still fill 148 SMs.  Each
// warp scores 4 rows per iteration (24 independent 16-byte loads in flight per
// lane), reduces with shuffles, and lane 0 appends (score,row) to a shared
// candidate buffer only if it is not worse than the CTA's running k-th best.
// The buffer is compacted with a block bitonic sort when it fills.  Per-split
// lists are merged by `topk_merge_kernel` (also the post-all-gather K4 merge).
// Roofline: HBM — 4*d bytes per candidate (no cross-query reuse assumed).
#include <math_constants.h>

#include "common.cuh"
#include "ptx.cuh"

namespace {

constexpr int RR_THREADS = 256;
constexpr int RR_WARPS = RR_THREADS / 32;
constexpr int RR_RPI = 4;                       // rows per warp iteration
constexpr int RR_ITERS = 4;                     // iterations per super-round
constexpr int RR_SUPER = RR_WARPS * RR_RPI * RR_ITERS;  // 128 rows between block syncs

struct RerankParams {
  const float* Q; int nq;
  const float* D; int64_t n; int d;
  const int64_t* leaf_offsets; int64_t n_leaves;
  const int32_t* leaf_docids;
  const int32_t* query_leaves; int L;
  int k; int cap;  // cap: power of two >= k + 2*RR_SUPER
  int S;
  int64_t id_base;
  float* out_scores; int64_t* out_ids;  // [nq*S, k]
  int32_t* n_candidates;
  int64_t max_rows;  // > 0: only the first max_rows candidate rows of every query (prefix of its leaf list)
  int* err_flag;     // set when a bounded pipeline wait times out (the top-k lists of that launch are then incomplete)
};

// after the launch sequence: a time-out must not leave a plausible but truncated result behind
__global__ void poison_topk_kernel(const int* __restrict__ err, float* __restrict__ scores, int64_t* __restrict__ ids, int64_t total) {
  if (*err == 0) return;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    scores[i] = __int_as_float(0x7fc00000);  // NaN
    ids[i] = -1;
  }
}

__device__ __forceinline__ void compact_buffer(float* s_score, int32_t* s_id, int* s_count, float* s_tau, int k, int cap) {
  __syncthreads();
  const int cnt = *s_count;
  for (int i = cnt + threadIdx.x; i < cap; i += blockDim.x) {
    s_score[i] = -CUDART_INF_F;
    s_id[i] = 0x7fffffff;
  }
  __syncthreads();
  block_bitonic_sort<int32_t>(s_score, s_id, cap);
  if (threadIdx.x == 0) {
    const int kept = cnt < k ? cnt : k;
    *s_count = kept;
    *s_tau = (kept >= k) ? s_score[k - 1] : -CUDART_INF_F;
  }
  __syncthreads();
}

template <int NCH>
__global__ void __launch_bounds__(RR_THREADS) rerank_kernel(RerankParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* s_score = reinterpret_cast<float*>(smem_raw);
  int32_t* s_id = reinterpret_cast<int32_t*>(s_score + p.cap);
  int64_t* s_prefix = reinterpret_cast<int64_t*>(s_id + p.cap);  // [L+1]
  int64_t* s_leafbeg = s_prefix + (p.L + 1);                     // [L]
  __shared__ int s_count;
  __shared__ float s_tau;

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t cta = blockIdx.x;
  const int q = (int)(cta / p.S);
  const int s = (int)(cta - (int64_t)q * p.S);
  const int d = p.d;

  // candidate prefix over this query's leaves (leaf order = beam order, main_models.py:3923)
  for (int t = threadIdx.x; t < p.L; t += RR_THREADS) {
    const int leaf = p.query_leaves[(int64_t)q * p.L + t];
    int64_t b = 0, sz = 0;
    if (leaf >= 0 && leaf < p.n_leaves) {
      b = p.leaf_offsets[leaf];
      sz = p.leaf_offsets[leaf + 1] - b;
    }
    s_leafbeg[t] = b;
    s_prefix[t + 1] = sz;
  }
  if (threadIdx.x == 0) {
    s_prefix[0] = 0;
    s_count = 0;
    s_tau = -CUDART_INF_F;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int64_t run = 0;
    for (int t = 1; t <= p.L; ++t) {
      run += s_prefix[t];
      s_prefix[t] = run;
    }
  }
  __syncthreads();
  const int64_t C = s_prefix[p.L];
  if (s == 0 && threadIdx.x == 0 && p.n_candidates) p.n_candidates[q] = (int32_t)(C > 0x7fffffff ? 0x7fffffff : C);
  const int64_t lo = C * s / p.S, hi = C * (s + 1) / p.S;

  float4 qreg[NCH];
#pragma unroll
  for (int t = 0; t < NCH; ++t) {
    int c4 = (lane + 32 * t) * 4;
    qreg[t] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c4 < d) qreg[t] = ldg_f4(p.Q + (int64_t)q * d + c4);
  }

  for (int64_t pos = lo; pos < hi; pos += RR_SUPER) {
#pragma unroll 1
    for (int it = 0; it < RR_ITERS; ++it) {
      const int64_t c0 = pos + (int64_t)(it * RR_WARPS + warp) * RR_RPI;
      if (c0 >= hi) break;
      // lanes 0..RPI-1 resolve candidate index -> row of D
      int32_t myrow = -1;
      if (lane < RR_RPI && c0 + lane < hi) {
        const int64_t ci = c0 + lane;
        int a = 0, b = p.L;  // find t with prefix[t] <= ci < prefix[t+1]
        while (b - a > 1) {
          int m = (a + b) >> 1;
          if (s_prefix[m] <= ci) a = m; else b = m;
        }
        myrow = p.leaf_docids[s_leafbeg[a] + (ci - s_prefix[a])];
      }
      int32_t rows[RR_RPI];
      float4 v[RR_RPI][NCH];
#pragma unroll
      for (int r = 0; r < RR_RPI; ++r) {
        rows[r] = __shfl_sync(MEVI_FULL_MASK, myrow, r);
        const float* src = p.D + (int64_t)(rows[r] < 0 ? 0 : rows[r]) * d;
#pragma unroll
        for (int t = 0; t < NCH; ++t) {
          int c4 = (lane + 32 * t) * 4;
          v[r][t] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (rows[r] >= 0 && c4 < d) v[r][t] = ld_stream_f4(src + c4);
        }
      }
#pragma unroll
      for (int r = 0; r < RR_RPI; ++r) {
        float acc = 0.f;
#pragma unroll
        for (int t = 0; t < NCH; ++t) {
          acc = fmaf(qreg[t].x, v[r][t].x, acc);
          acc = fmaf(qreg[t].y, v[r][t].y, acc);
          acc = fmaf(qreg[t].z, v[r][t].z, acc);
          acc = fmaf(qreg[t].w, v[r][t].w, acc);
        }
        acc = warp_sum(acc);
        if (lane == 0 && rows[r] >= 0) {
          const float tau = *reinterpret_cast<volatile float*>(&s_tau);
          if (!(acc < tau)) {
            const int slot = atomicAdd(&s_count, 1);
            s_score[slot] = acc;  // slot < cap: at most RR_SUPER appends between compactions
            s_id[slot] = rows[r];
          }
        }
      }
    }
    __syncthreads();
    if (s_count > p.cap - RR_SUPER) compact_buffer(s_score, s_id, &s_count, &s_tau, p.k, p.cap);
  }
  compact_buffer(s_score, s_id, &s_count, &s_tau, p.k, p.cap);
  const int kept = s_count;
  float* os = p.out_scores + cta * p.k;
  int64_t* oi = p.out_ids + cta * p.k;
  for (int i = threadIdx.x; i < p.k; i += RR_THREADS) {
    if (i < kept) {
      os[i] = s_score[i];
      oi[i] = p.id_base + (int64_t)s_id[i];
    } else {
      os[i] = -CUDART_INF_F;
      oi[i] = -1;
    }
  }
}


// ---- leaf-ordered streaming variant ---------------------------------------------------------------
// D is stored in CSR (leaf) order, so a leaf is one contiguous byte range: candidates are streamed with
// bulk async copies (TMA engine) into a shared-memory ring by a producer warp — no registers tied up in
// flight, six 8-row stages (144 KB at d=768) of loads outstanding per SM, one TLB page per leaf instead
// of one per candidate.  Eight consumer warps take one row each per stage (conflict-free 16 B shared
// loads), reduce with shuffles and feed the same threshold + bitonic-compaction top-k as above.
constexpr int RS_ROWS = 8;      // rows per stage (one per consumer warp)
constexpr int RS_STAGES = 6;
constexpr int RS_CONSUMERS = 8; // warps 1..8; warp 0 is the producer
constexpr int RS_THREADS = 32 * (1 + RS_CONSUMERS);
constexpr int RS_CHECK = 16;    // stages between compaction checks (<= 128 appends)
constexpr int RS_OCC_SLOT = 512;  // multi-cluster: the stage's rows of the occurrence table (<= 8 x 15 int32, 16 B aligned)

__device__ __forceinline__ void consumer_bar() { asm volatile("bar.sync 1, %0;" ::"n"(32 * RS_CONSUMERS) : "memory"); }

// --doc_multiclus > 1 (main_models.py:3998-4011): a document listed under several leaves has several CSR positions.
// occ_leaves [n, C-1] int32 holds, per CSR position, the leaves of the document's OTHER positions (-1 padded; -2 - leaf
// for an earlier position in the same leaf, when a leaf lists the document more than once).  Per
// (query, document) exactly one occurrence is kept, the canonical one: the first position of the query's leaf list whose
// leaf lists the document (and the first CSR position inside that leaf).  It is scored agg(c, s), c = the number of positions of the leaf list that list the document.
struct MultiClus {
  const int32_t* occ_leaves;
  int C;         // largest number of positions of any document (1 <= C <= 16)
  int aggr;      // MEVI_MULTICLUS_ADD / _MAX
  int hash_log2; // the per-CTA leaf table has 1 << hash_log2 >= 2L slots
};

__device__ __forceinline__ int leaf_slot(const int32_t* s_hkey, int leaf, int hash_log2) {
  const unsigned mask = (1u << hash_log2) - 1u;
  unsigned h = ((unsigned)leaf * 0x9E3779B1u) >> (32 - hash_log2);
  for (;;) {  // load factor <= 1/2: a free slot ends every probe sequence
    const int k = s_hkey[h];
    if (k == leaf) return (int)h;
    if (k < 0) return -1;
    h = (h + 1) & mask;
  }
}

template <int NCH, bool MC>
__device__ __forceinline__ void rerank_stream_body(const RerankParams& p, const MultiClus& mc) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int d = p.d;
  const uint32_t row_bytes = (uint32_t)d * 4u;
  const uint32_t stage_bytes = RS_ROWS * row_bytes;
  unsigned char* s_ring = smem_raw;                                                  // [RS_STAGES][RS_ROWS][d] fp32
  unsigned char* s_occ = s_ring + (size_t)RS_STAGES * stage_bytes;                    // MC: [RS_STAGES][RS_OCC_SLOT]
  float* s_score = reinterpret_cast<float*>(s_occ + (MC ? RS_STAGES * RS_OCC_SLOT : 0));
  int32_t* s_id = reinterpret_cast<int32_t*>(s_score + p.cap);
  int64_t* s_prefix = reinterpret_cast<int64_t*>(s_id + p.cap);                      // [L+1]
  int64_t* s_leafbeg = s_prefix + (p.L + 1);                                         // [L]
  // MC: open-addressed table of the query's leaves -> first position in its leaf list, number of positions; and per
  // position t its leaf's number of positions when t is that leaf's first position, else -1 (a repeated leaf)
  int32_t* s_hkey = reinterpret_cast<int32_t*>(s_leafbeg + p.L);                     // [1 << hash_log2]
  int32_t* s_hfirst = s_hkey + (MC ? (1 << mc.hash_log2) : 0);
  int32_t* s_hmult = s_hfirst + (MC ? (1 << mc.hash_log2) : 0);
  int32_t* s_own = s_hmult + (MC ? (1 << mc.hash_log2) : 0);                          // [L]
  __shared__ __align__(8) uint64_t full_bar[RS_STAGES];
  __shared__ __align__(8) uint64_t empty_bar[RS_STAGES];
  __shared__ int s_meta_row[RS_STAGES];
  __shared__ int s_meta_n[RS_STAGES];
  __shared__ int s_count;
  __shared__ float s_tau;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t cta = blockIdx.x;
  const int q = (int)(cta / p.S);
  const int s = (int)(cta - (int64_t)q * p.S);

  for (int t = tid; t < p.L; t += RS_THREADS) {
    const int leaf = p.query_leaves[(int64_t)q * p.L + t];
    int64_t b = 0, sz = 0;
    if (leaf >= 0 && leaf < p.n_leaves) {
      b = p.leaf_offsets[leaf];
      sz = p.leaf_offsets[leaf + 1] - b;
    }
    s_leafbeg[t] = b;
    s_prefix[t + 1] = sz;
  }
  if constexpr (MC) {
    for (int i = tid; i < (1 << mc.hash_log2); i += RS_THREADS) {
      s_hkey[i] = -1;
      s_hfirst[i] = 0x7fffffff;
      s_hmult[i] = 0;
    }
  }
  if (tid == 0) {
    s_prefix[0] = 0;
    s_count = 0;
    s_tau = -CUDART_INF_F;
    for (int i = 0; i < RS_STAGES; ++i) {
      ptx::mbar_init(&full_bar[i], 1);
      ptx::mbar_init(&empty_bar[i], RS_CONSUMERS);
    }
    ptx::mbar_fence_init();
  }
  __syncthreads();
  if constexpr (MC) {  // (before the scan below overwrites the leaf sizes)
    for (int t = tid; t < p.L; t += RS_THREADS) {
      if (s_prefix[t + 1] == 0) continue;  // no document: never streamed, never a sibling
      const int leaf = p.query_leaves[(int64_t)q * p.L + t];
      const unsigned mask = (1u << mc.hash_log2) - 1u;
      unsigned h = ((unsigned)leaf * 0x9E3779B1u) >> (32 - mc.hash_log2);
      for (;;) {
        const int prev = atomicCAS(&s_hkey[h], -1, leaf);
        if (prev < 0 || prev == leaf) break;
        h = (h + 1) & mask;
      }
      atomicMin(&s_hfirst[h], t);
      atomicAdd(&s_hmult[h], 1);
    }
    __syncthreads();
  }
  if (tid == 0) {
    int64_t run = 0;
    for (int t = 1; t <= p.L; ++t) {
      run += s_prefix[t];
      s_prefix[t] = run;
    }
  }
  __syncthreads();
  if constexpr (MC) {
    for (int t = tid; t < p.L; t += RS_THREADS) {
      int own = -1;
      if (s_prefix[t + 1] > s_prefix[t]) {
        const int h = leaf_slot(s_hkey, p.query_leaves[(int64_t)q * p.L + t], mc.hash_log2);
        if (s_hfirst[h] == t) own = s_hmult[h];
      }
      s_own[t] = own;
    }
    __syncthreads();
  }
  int64_t C = s_prefix[p.L];
  if (s == 0 && tid == 0 && p.n_candidates) p.n_candidates[q] = (int32_t)(C > 0x7fffffff ? 0x7fffffff : C);
  if (p.max_rows > 0 && C > p.max_rows) C = p.max_rows;
  const int64_t lo = C * s / p.S, hi = C * (s + 1) / p.S;

  if (warp == 0) {
    // ===== producer =====
    if (lane == 0) {
      uint32_t g = 0;
      bool ok = true;
      for (int t = 0; t < p.L && ok; ++t) {
        int64_t a = s_prefix[t] > lo ? s_prefix[t] : lo;
        const int64_t b = s_prefix[t + 1] < hi ? s_prefix[t + 1] : hi;
        for (; a < b && ok; a += RS_ROWS, ++g) {
          const int nrows = (int)((b - a) < RS_ROWS ? (b - a) : RS_ROWS);
          const int64_t row = s_leafbeg[t] + (a - s_prefix[t]);
          const uint32_t st = g % RS_STAGES, ph = (g / RS_STAGES) & 1;
          if (!ptx::mbar_wait(&empty_bar[st], ph ^ 1)) { atomicExch(p.err_flag, 1); ok = false; break; }
          s_meta_row[st] = (int)row;
          s_meta_n[st] = MC ? (nrows | (t << 4)) : nrows;  // MC: the leaf's position in the query's list rides along
          const uint32_t bytes = (uint32_t)nrows * row_bytes;
          uint32_t occ_bytes = 0;
          int64_t occ0 = 0;
          if constexpr (MC) {  // the rows' slice of the occurrence table travels with them, widened to 16 B bounds
            const int64_t w4 = (int64_t)(mc.C - 1) * 4;
            occ0 = (row * w4) & ~int64_t(15);
            occ_bytes = (uint32_t)((((row + nrows) * w4 + 15) & ~int64_t(15)) - occ0);
          }
          ptx::mbar_arrive_expect_tx(&full_bar[st], bytes + occ_bytes);
          ptx::bulk_g2s(s_ring + (size_t)st * stage_bytes, p.D + row * d, bytes, &full_bar[st]);
          if (occ_bytes)
            ptx::bulk_g2s(s_occ + st * RS_OCC_SLOT, reinterpret_cast<const char*>(mc.occ_leaves) + occ0, occ_bytes, &full_bar[st]);
        }
      }
      // sentinel: tells the consumers the stream has ended
      const uint32_t st = g % RS_STAGES, ph = (g / RS_STAGES) & 1;
      if (ok) {
        if (ptx::mbar_wait(&empty_bar[st], ph ^ 1)) {
          s_meta_n[st] = 0;
          ptx::mbar_arrive(&full_bar[st]);
        } else {
          atomicExch(p.err_flag, 2);
        }
      }
    }
  } else {
    // ===== consumers =====
    const int cw = warp - 1;
    const int gtid = tid - 32;
    float4 qreg[NCH];
#pragma unroll
    for (int t = 0; t < NCH; ++t) {
      const int c4 = (lane + 32 * t) * 4;
      qreg[t] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c4 < d) qreg[t] = ldg_f4(p.Q + (int64_t)q * d + c4);
    }
    uint32_t g = 0;
    for (;; ++g) {
      const uint32_t st = g % RS_STAGES, ph = (g / RS_STAGES) & 1;
      if (!ptx::mbar_wait(&full_bar[st], ph)) { atomicExch(p.err_flag, 3); break; }
      const int meta = s_meta_n[st];
      const int nrows = MC ? (meta & 15) : meta;
      if (nrows == 0) break;
      if (cw < nrows) {
        const float* src = reinterpret_cast<const float*>(s_ring + (size_t)st * stage_bytes + (size_t)cw * row_bytes);
        int32_t sib = -1;
        if constexpr (MC) {
          if (lane >= 1 && lane < mc.C) {
            const int64_t w = mc.C - 1, row0 = s_meta_row[st];
            const int64_t e = (row0 + cw) * w + (lane - 1) - (((row0 * w * 4) & ~int64_t(15)) >> 2);
            sib = reinterpret_cast<const int32_t*>(s_occ + st * RS_OCC_SLOT)[e];
          }
        }
        float acc = 0.f;
#pragma unroll
        for (int t = 0; t < NCH; ++t) {
          const int c4 = (lane + 32 * t) * 4;
          if (c4 < d) {
            const float4 v = *reinterpret_cast<const float4*>(src + c4);
            acc = fmaf(qreg[t].x, v.x, acc);
            acc = fmaf(qreg[t].y, v.y, acc);
            acc = fmaf(qreg[t].z, v.z, acc);
            acc = fmaf(qreg[t].w, v.w, acc);
          }
        }
        acc = warp_sum(acc);
        bool keep = true;
        if constexpr (MC) {
          // lane 0: this position's own leaf; lanes 1..C-1: the leaves of the document's other positions.  The occurrence
          // is canonical when no leaf of the document comes earlier in the query's list.
          const int t = meta >> 4;
          int mult = 0;
          bool earlier = false;
          if (lane == 0) {
            mult = s_own[t];
            earlier = mult < 0;
          } else if (sib <= -2) {  // the document also sits at an earlier position of this same leaf
            earlier = true;
          } else if (sib >= 0) {
            const int h = leaf_slot(s_hkey, sib, mc.hash_log2);
            if (h >= 0) {
              mult = s_hmult[h];
              earlier = s_hfirst[h] < t;
            }
          }
          keep = __ballot_sync(MEVI_FULL_MASK, earlier) == 0u;
          const int c = __reduce_add_sync(MEVI_FULL_MASK, earlier ? 0 : mult);
          if (keep && mc.aggr == MEVI_MULTICLUS_ADD) {
            float a = 0.f;  // the reference's fold: zeros, then += s once per position (main_models.py:4004-4007)
            for (int i = 0; i < c; ++i) a = __fadd_rn(a, acc);
            acc = a;
          }
        }
        if (lane == 0 && keep) {
          const float tau = *reinterpret_cast<volatile float*>(&s_tau);
          if (!(acc < tau)) {
            const int slot = atomicAdd(&s_count, 1);
            s_score[slot] = acc;
            s_id[slot] = p.leaf_docids[s_meta_row[st] + cw];  // CSR position -> document row
          }
        }
      }
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&empty_bar[st]);
      if ((g % RS_CHECK) == RS_CHECK - 1) {
        consumer_bar();
        const int cnt = s_count;
        if (cnt > p.cap - RS_CHECK * RS_ROWS) {
          for (int i = cnt + gtid; i < p.cap; i += 32 * RS_CONSUMERS) {
            s_score[i] = -CUDART_INF_F;
            s_id[i] = 0x7fffffff;
          }
          consumer_bar();
          group_bitonic_sort<int32_t>(s_score, s_id, p.cap, gtid, 32 * RS_CONSUMERS, 1);
          if (gtid == 0) {
            const int kept = cnt < p.k ? cnt : p.k;
            s_count = kept;
            s_tau = (kept >= p.k) ? s_score[p.k - 1] : -CUDART_INF_F;
          }
        }
        consumer_bar();
      }
    }
    // final compaction + output
    consumer_bar();
    const int cnt = s_count;
    for (int i = cnt + gtid; i < p.cap; i += 32 * RS_CONSUMERS) {
      s_score[i] = -CUDART_INF_F;
      s_id[i] = 0x7fffffff;
    }
    consumer_bar();
    group_bitonic_sort<int32_t>(s_score, s_id, p.cap, gtid, 32 * RS_CONSUMERS, 1);
    const int kept = cnt < p.k ? cnt : p.k;
    float* os = p.out_scores + cta * p.k;
    int64_t* oi = p.out_ids + cta * p.k;
    for (int i = gtid; i < p.k; i += 32 * RS_CONSUMERS) {
      if (i < kept) {
        os[i] = s_score[i];
        oi[i] = p.id_base + (int64_t)s_id[i];
      } else {
        os[i] = -CUDART_INF_F;
        oi[i] = -1;
      }
    }
  }
}

template <int NCH>
__global__ void __launch_bounds__(RS_THREADS) rerank_stream_kernel(RerankParams p) {
  rerank_stream_body<NCH, false>(p, MultiClus{});
}

template <int NCH>
__global__ void __launch_bounds__(RS_THREADS) rerank_stream_multiclus_kernel(RerankParams p, MultiClus mc) {
  rerank_stream_body<NCH, true>(p, mc);
}

template <int NCH>
cudaError_t launch_rerank_stream(const RerankParams& p, const MultiClus* mc, size_t smem, cudaStream_t st) {
  const int64_t grid = (int64_t)p.nq * p.S;
  if (mc) {
    cudaError_t e = cudaFuncSetAttribute(rerank_stream_multiclus_kernel<NCH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    rerank_stream_multiclus_kernel<NCH><<<(unsigned)grid, RS_THREADS, smem, st>>>(p, *mc);
    return cudaGetLastError();
  }
  cudaError_t e = cudaFuncSetAttribute(rerank_stream_kernel<NCH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  rerank_stream_kernel<NCH><<<(unsigned)grid, RS_THREADS, smem, st>>>(p);
  return cudaGetLastError();
}

__global__ void gather_rows_kernel(const float* __restrict__ D, int d4, const int32_t* __restrict__ rows, int64_t m,
                                   float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t warp_global = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t i = warp_global; i < m; i += n_warps) {
    const float4* src = reinterpret_cast<const float4*>(D) + (int64_t)rows[i] * d4;
    float4* dst = reinterpret_cast<float4*>(out) + i * d4;
    for (int c = lane; c < d4; c += 32) dst[c] = __ldg(src + c);
  }
}

// One CTA per query: merge S lists of k (score,id) into the k best. cap = pow2 >= S*k.
__global__ void __launch_bounds__(256) topk_merge_kernel(const float* __restrict__ in_s, const int64_t* __restrict__ in_i,
                                                         int S, int nq, int k, int cap, int64_t list_stride,
                                                         int64_t shard_stride, float* __restrict__ out_s,
                                                         int64_t* __restrict__ out_i) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  int64_t* s_id = reinterpret_cast<int64_t*>(smem_raw);
  float* s_score = reinterpret_cast<float*>(s_id + cap);
  const int q = blockIdx.x;
  const int total = S * k;
  for (int i = threadIdx.x; i < cap; i += blockDim.x) {
    if (i < total) {
      const int sh = i / k, j = i - sh * k;
      const int64_t src = (int64_t)sh * shard_stride + (int64_t)q * list_stride + j;
      float sc = in_s[src];
      int64_t id = in_i[src];
      if (id < 0) {  // padding from a shard that held fewer than k candidates
        sc = -CUDART_INF_F;
        id = INT64_MAX;
      }
      s_score[i] = sc;
      s_id[i] = id;
    } else {
      s_score[i] = -CUDART_INF_F;
      s_id[i] = INT64_MAX;
    }
  }
  __syncthreads();
  block_bitonic_sort<int64_t>(s_score, s_id, cap);
  for (int i = threadIdx.x; i < k; i += blockDim.x) {
    const bool pad = (s_id[i] == INT64_MAX);
    out_s[(int64_t)q * k + i] = pad ? -CUDART_INF_F : s_score[i];
    out_i[(int64_t)q * k + i] = pad ? -1 : s_id[i];
  }
}

// Every candidate's score, no top-k: the output mode of the shipped re-rank recipe (`--save_hard_neg 8841823`,
// MEVI/main_models.py:4012-4014, 4046-4053 keeps ALL candidates, sorted).  Leaf-ordered layout; candidate position pos
// of query q (leaf order = beam order, then row order inside the leaf - the reference's concatenation order, 3994-3997)
// goes to out[out_offsets[q] + pos].  One warp per row, summation order of the dense scorer; the caller sorts.
template <int NCH>
__global__ void __launch_bounds__(256) rerank_all_kernel(RerankParams p, const int64_t* __restrict__ out_offsets) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  int64_t* s_prefix = reinterpret_cast<int64_t*>(smem_raw);  // [L+1]
  int64_t* s_leafbeg = s_prefix + (p.L + 1);                 // [L]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int q = (int)(blockIdx.x / p.S), s = (int)(blockIdx.x - (int64_t)q * p.S);
  const int d = p.d;
  for (int t = threadIdx.x; t < p.L; t += blockDim.x) {
    const int leaf = p.query_leaves[(int64_t)q * p.L + t];
    int64_t b = 0, sz = 0;
    if (leaf >= 0 && leaf < p.n_leaves) {
      b = p.leaf_offsets[leaf];
      sz = p.leaf_offsets[leaf + 1] - b;
    }
    s_leafbeg[t] = b;
    s_prefix[t + 1] = sz;
  }
  if (threadIdx.x == 0) s_prefix[0] = 0;
  __syncthreads();
  if (threadIdx.x == 0) {
    int64_t run = 0;
    for (int t = 1; t <= p.L; ++t) {
      run += s_prefix[t];
      s_prefix[t] = run;
    }
  }
  __syncthreads();
  const int64_t C = s_prefix[p.L];
  if (s == 0 && threadIdx.x == 0 && p.n_candidates) p.n_candidates[q] = (int32_t)(C > 0x7fffffff ? 0x7fffffff : C);
  const int64_t lo = C * s / p.S, hi = C * (s + 1) / p.S;
  const int64_t obase = out_offsets[q];
  float4 qreg[NCH];
#pragma unroll
  for (int t = 0; t < NCH; ++t) {
    const int c4 = (lane + 32 * t) * 4;
    qreg[t] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c4 < d) qreg[t] = ldg_f4(p.Q + (int64_t)q * d + c4);
  }
  int t_cur = 0;
  for (int64_t pos = lo + warp; pos < hi; pos += 8) {
    while (s_prefix[t_cur + 1] <= pos) ++t_cur;  // pos only grows: the leaf cursor moves forward
    const int64_t row = s_leafbeg[t_cur] + (pos - s_prefix[t_cur]);
    const float* src = p.D + row * d;
    float4 v[NCH];
#pragma unroll
    for (int t = 0; t < NCH; ++t) {
      const int c4 = (lane + 32 * t) * 4;
      v[t] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c4 < d) v[t] = ld_stream_f4(src + c4);
    }
    float acc = 0.f;
#pragma unroll
    for (int t = 0; t < NCH; ++t) {
      acc = fmaf(qreg[t].x, v[t].x, acc);
      acc = fmaf(qreg[t].y, v[t].y, acc);
      acc = fmaf(qreg[t].z, v[t].z, acc);
      acc = fmaf(qreg[t].w, v[t].w, acc);
    }
    acc = warp_sum(acc);
    if (lane == 0) {
      p.out_scores[obase + pos] = acc;
      p.out_ids[obase + pos] = p.id_base + (int64_t)p.leaf_docids[row];
    }
  }
}

template <int NCH>
cudaError_t launch_rerank_all(const RerankParams& p, const int64_t* out_offsets, size_t smem, cudaStream_t st) {
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(rerank_all_kernel<NCH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  rerank_all_kernel<NCH><<<(unsigned)((int64_t)p.nq * p.S), 256, smem, st>>>(p, out_offsets);
  return cudaGetLastError();
}

int next_pow2(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

template <int NCH>
cudaError_t launch_rerank(const RerankParams& p, size_t smem, cudaStream_t st) {
  cudaError_t e = cudaFuncSetAttribute(rerank_kernel<NCH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const int64_t grid = (int64_t)p.nq * p.S;
  rerank_kernel<NCH><<<(unsigned)grid, RR_THREADS, smem, st>>>(p);
  return cudaGetLastError();
}

}  // namespace

// internal: merge with explicit strides (used by re-rank splits and the public merge)
int mevi_topk_merge_launch(mevi_ctx* ctx, const float* in_s, const int64_t* in_i, int S, int nq, int k,
                           int64_t list_stride, int64_t shard_stride, float* out_s, int64_t* out_i, cudaStream_t st) {
  const int cap = next_pow2(S * k);
  MEVI_REQUIRE(ctx, cap <= 16384, "top-k merge of %d lists x k=%d exceeds the 16384-entry shared-memory sorter", S, k);
  const size_t smem = (size_t)cap * (sizeof(int64_t) + sizeof(float));
  MEVI_CUDA(ctx, cudaFuncSetAttribute(topk_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  topk_merge_kernel<<<nq, 256, smem, st>>>(in_s, in_i, S, nq, k, cap, list_stride, shard_stride, out_s, out_i);
  MEVI_COUNT_LAUNCH(ctx, 1);
  MEVI_CUDA(ctx, cudaGetLastError());
  return MEVI_OK;
}

extern "C" {

static int cluster_rerank_impl(mevi_ctx* ctx, const float* Q, int nq, const float* D, int64_t n, int d, int d_layout,
                               const int64_t* leaf_offsets, int64_t n_leaves, const int32_t* leaf_docids,
                               const int32_t* query_leaves, int L, int k, int64_t id_base, float* scores, int64_t* ids,
                               int32_t* n_candidates, int64_t max_rows, const MultiClus* mc, void* stream);

int mevi_cluster_rerank(mevi_ctx* ctx, const float* Q, int nq, const float* D, int64_t n, int d, int d_layout,
                        const int64_t* leaf_offsets, int64_t n_leaves, const int32_t* leaf_docids,
                        const int32_t* query_leaves, int L, int k, int64_t id_base, float* scores, int64_t* ids,
                        int32_t* n_candidates, void* stream) {
  return cluster_rerank_impl(ctx, Q, nq, D, n, d, d_layout, leaf_offsets, n_leaves, leaf_docids, query_leaves, L, k, id_base,
                             scores, ids, n_candidates, 0, nullptr, stream);
}

// Same, restricted to the first max_rows candidate rows of every query (leaf-ordered layout only): the exact top-k
// of a prefix of the candidates.  Its k-th score is a lower bound of the query's final k-th score — the starting
// threshold of the grouped re-rank (mevi_rerank_grouped_begin).
int mevi_cluster_rerank_prefix(mevi_ctx* ctx, const float* Q, int nq, const float* D_leaf, int64_t n, int d,
                               const int64_t* leaf_offsets, int64_t n_leaves, const int32_t* leaf_docids,
                               const int32_t* query_leaves, int L, int k, int64_t max_rows, float* scores, int64_t* ids,
                               int32_t* n_candidates, void* stream) {
  if (ctx && max_rows <= 0) return mevi_set_error(ctx, MEVI_ERR_INVALID, "max_rows must be positive");
  return cluster_rerank_impl(ctx, Q, nq, D_leaf, n, d, 1, leaf_offsets, n_leaves, leaf_docids, query_leaves, L, k, 0, scores, ids,
                             n_candidates, max_rows, nullptr, stream);
}

// --doc_multiclus > 1: one entry per (query, document), its score aggregated over the query's leaves that list it.
int mevi_cluster_rerank_multiclus(mevi_ctx* ctx, const float* Q, int nq, const float* D_leaf, int64_t n, int d,
                                  const int64_t* leaf_offsets, int64_t n_leaves, const int32_t* leaf_docids,
                                  const int32_t* occ_leaves, int C, const int32_t* query_leaves, int L, int k, int aggr,
                                  int64_t id_base, float* scores, int64_t* ids, int32_t* n_candidates, void* stream) {
  MEVI_CHECK_CTX(ctx);
  MEVI_REQUIRE(ctx, aggr == MEVI_MULTICLUS_ADD || aggr == MEVI_MULTICLUS_MAX, "aggr must be MEVI_MULTICLUS_ADD or _MAX (got %d)", aggr);
  MEVI_REQUIRE(ctx, C >= 1 && (C == 1 || occ_leaves), "C must be >= 1, with an occurrence table when C > 1");
  MEVI_REQUIRE(ctx, ((uintptr_t)occ_leaves & 15) == 0, "occ_leaves must be 16-byte aligned");
  if (C > 16)
    return mevi_set_error(ctx, MEVI_ERR_UNSUPPORTED, "multi-cluster re-rank: a document is listed under %d leaves (at most 16)", C);
  MultiClus mc;
  mc.occ_leaves = occ_leaves;
  mc.C = C;
  mc.aggr = aggr;
  mc.hash_log2 = 1;
  while ((1 << mc.hash_log2) < 2 * L) ++mc.hash_log2;
  return cluster_rerank_impl(ctx, Q, nq, D_leaf, n, d, 1, leaf_offsets, n_leaves, leaf_docids, query_leaves, L, k, id_base, scores,
                             ids, n_candidates, 0, &mc, stream);
}

static int cluster_rerank_impl(mevi_ctx* ctx, const float* Q, int nq, const float* D, int64_t n, int d, int d_layout,
                               const int64_t* leaf_offsets, int64_t n_leaves, const int32_t* leaf_docids,
                               const int32_t* query_leaves, int L, int k, int64_t id_base, float* scores, int64_t* ids,
                               int32_t* n_candidates, int64_t max_rows, const MultiClus* mc, void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  MEVI_REQUIRE(ctx, Q && D && leaf_offsets && leaf_docids && query_leaves && scores && ids, "NULL argument");
  MEVI_REQUIRE(ctx, d > 0 && d % 4 == 0 && d <= 1024, "re-rank needs d %% 4 == 0 and d <= 1024 (got %d)", d);
  MEVI_REQUIRE(ctx, k >= 1 && k <= 2048, "k must be in [1, 2048] (got %d)", k);
  MEVI_REQUIRE(ctx, L >= 1 && L <= 4096, "L must be in [1, 4096] (got %d)", L);
  MEVI_REQUIRE(ctx, n < (int64_t)2147483647, "shard too large for int32 row ids");
  if (nq <= 0) return MEVI_OK;
  if (int rc = mevi_deferred_error(ctx)) return rc;
  MEVI_REQUIRE(ctx, d_layout == 0 || d_layout == 1, "d_layout must be 0 (document order) or 1 (CSR / leaf order)");
  const int cap = next_pow2(k + 2 * RR_SUPER);
  int S = (4 * ctx->sm_count + nq - 1) / nq;
  const int smax = 8192 / next_pow2(k) < 64 ? 8192 / next_pow2(k) : 64;
  if (S > smax) S = smax;
  if (S < 1) S = 1;
  MEVI_REQUIRE(ctx, (int64_t)nq * S < (int64_t)2147483647, "too many (query, split) CTAs");
  RerankParams p;
  p.Q = Q; p.nq = nq; p.D = D; p.n = n; p.d = d;
  p.leaf_offsets = leaf_offsets; p.n_leaves = n_leaves; p.leaf_docids = leaf_docids;
  p.query_leaves = query_leaves; p.L = L; p.k = k; p.cap = cap; p.S = S; p.id_base = id_base;
  p.n_candidates = n_candidates;
  p.max_rows = max_rows;
  p.err_flag = ctx->dev_err + MEVI_ERRSLOT_RERANK;
  if (S == 1) {
    p.out_scores = scores;
    p.out_ids = ids;
  } else {
    size_t bytes = (size_t)nq * S * k * (sizeof(float) + sizeof(int64_t));
    char* ws = (char*)mevi_ws(ctx, WS_TOPK_PART, bytes);
    if (!ws) return MEVI_ERR_NOMEM;
    p.out_ids = (int64_t*)ws;
    p.out_scores = (float*)(ws + (size_t)nq * S * k * sizeof(int64_t));
  }
  size_t smem = (size_t)cap * 8 + (size_t)(2 * L + 1) * sizeof(int64_t);
  if (mc) smem += (size_t)(3 * (1 << mc->hash_log2) + L) * sizeof(int32_t) + RS_STAGES * RS_OCC_SLOT;  // leaf table, own-leaf counts, table slices
  cudaError_t e;
  const size_t ring = (size_t)RS_STAGES * RS_ROWS * d * 4;
  if (d_layout == 1 && smem + ring + 256 <= 220 * 1024) {
    smem += ring + 128;
    if (d <= 128) e = launch_rerank_stream<1>(p, mc, smem, st);
    else if (d <= 256) e = launch_rerank_stream<2>(p, mc, smem, st);
    else if (d <= 512) e = launch_rerank_stream<4>(p, mc, smem, st);
    else if (d <= 768) e = launch_rerank_stream<6>(p, mc, smem, st);
    else e = launch_rerank_stream<8>(p, mc, smem, st);
  } else if (d_layout == 1) {
    return mevi_set_error(ctx, MEVI_ERR_UNSUPPORTED, "leaf-ordered re-rank: ring + top-k buffers exceed shared memory (d=%d k=%d L=%d)", d, k, L);
  } else if (d <= 128) e = launch_rerank<1>(p, smem, st);
  else if (d <= 256) e = launch_rerank<2>(p, smem, st);
  else if (d <= 512) e = launch_rerank<4>(p, smem, st);
  else if (d <= 768) e = launch_rerank<6>(p, smem, st);
  else e = launch_rerank<8>(p, smem, st);
  if (e != cudaSuccess) return mevi_set_error(ctx, MEVI_ERR_CUDA, "rerank launch: %s", cudaGetErrorString(e));
  MEVI_COUNT_LAUNCH(ctx, 1);
  if (S > 1) {
    // lists of one query are contiguous: [q][s][k]  -> shard_stride = k, list_stride = S*k
    int rc = mevi_topk_merge_launch(ctx, p.out_scores, p.out_ids, S, nq, k, (int64_t)S * k, (int64_t)k, scores, ids, st);
    if (rc != MEVI_OK) return rc;
  }
  poison_topk_kernel<<<ctx->sm_count, 256, 0, st>>>(p.err_flag, scores, ids, (int64_t)nq * k);
  MEVI_COUNT_LAUNCH(ctx, 1);
  return mevi_publish_errors(ctx, st);
}

int mevi_cluster_rerank_all(mevi_ctx* ctx, const float* Q, int nq, const float* D_leaf, int64_t n, int d,
                            const int64_t* leaf_offsets, int64_t n_leaves, const int32_t* leaf_docids,
                            const int32_t* query_leaves, int L, int64_t id_base, const int64_t* out_offsets, float* scores,
                            int64_t* ids, int32_t* n_candidates, void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  MEVI_REQUIRE(ctx, Q && D_leaf && leaf_offsets && leaf_docids && query_leaves && out_offsets && scores && ids, "NULL argument");
  MEVI_REQUIRE(ctx, d > 0 && d % 4 == 0 && d <= 1024, "re-rank needs d %% 4 == 0 and d <= 1024 (got %d)", d);
  MEVI_REQUIRE(ctx, L >= 1 && L <= 4096, "L must be in [1, 4096] (got %d)", L);
  if (nq <= 0) return MEVI_OK;
  int S = (8 * ctx->sm_count + nq - 1) / nq;
  if (S < 1) S = 1;
  if (S > 256) S = 256;
  RerankParams p;
  p.Q = Q; p.nq = nq; p.D = D_leaf; p.n = n; p.d = d;
  p.leaf_offsets = leaf_offsets; p.n_leaves = n_leaves; p.leaf_docids = leaf_docids;
  p.query_leaves = query_leaves; p.L = L; p.k = 0; p.cap = 0; p.S = S; p.id_base = id_base;
  p.out_scores = scores; p.out_ids = ids; p.n_candidates = n_candidates; p.max_rows = 0;
  p.err_flag = ctx->dev_err + MEVI_ERRSLOT_RERANK;
  const size_t smem = (size_t)(2 * L + 1) * sizeof(int64_t);
  cudaError_t e;
  if (d <= 128) e = launch_rerank_all<1>(p, out_offsets, smem, st);
  else if (d <= 256) e = launch_rerank_all<2>(p, out_offsets, smem, st);
  else if (d <= 512) e = launch_rerank_all<4>(p, out_offsets, smem, st);
  else if (d <= 768) e = launch_rerank_all<6>(p, out_offsets, smem, st);
  else e = launch_rerank_all<8>(p, out_offsets, smem, st);
  if (e != cudaSuccess) return mevi_set_error(ctx, MEVI_ERR_CUDA, "rerank_all launch: %s", cudaGetErrorString(e));
  MEVI_COUNT_LAUNCH(ctx, 1);
  return MEVI_OK;
}

int mevi_gather_rows(mevi_ctx* ctx, const float* D, int64_t n, int d, const int32_t* rows, int64_t m, float* out,
                     void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  MEVI_REQUIRE(ctx, D && rows && out && d > 0 && d % 4 == 0 && n >= 0 && m >= 0, "bad argument");
  if (m == 0) return MEVI_OK;
  gather_rows_kernel<<<ctx->sm_count * 8, 256, 0, (cudaStream_t)stream>>>(D, d / 4, rows, m, out);
  MEVI_CUDA(ctx, cudaGetLastError());
  MEVI_COUNT_LAUNCH(ctx, 1);
  return MEVI_OK;
}

int mevi_topk_merge(mevi_ctx* ctx, const float* scores_in, const int64_t* ids_in, int S, int nq, int k, float* scores,
                    int64_t* ids, void* stream) {
  MEVI_CHECK_CTX(ctx);
  DeviceGuard g(ctx->device);
  MEVI_REQUIRE(ctx, scores_in && ids_in && scores && ids && S >= 1 && nq >= 0 && k >= 1, "bad argument");
  if (nq == 0) return MEVI_OK;
  return mevi_topk_merge_launch(ctx, scores_in, ids_in, S, nq, k, (int64_t)k, (int64_t)nq * k, scores, ids,
                                (cudaStream_t)stream);
}

}  // extern "C"
