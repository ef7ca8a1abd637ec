// search.cu — flat inner-product top-k search on sm_100a.
//
// Replaces faiss.IndexFlatIP(dim).add / .search as called by the reference at
//   drivers/run_ann_data_gen.py:269-276,303 and drivers/run_ann_data_gen_dpr.py:238-252.
//
// Pipeline of one ance_index_search (all on the caller's stream):
//   1. quantize_rows_kernel : Q fp32 -> 16-bit operands (+ ||q^||, ||q - q^|| per query)
//   2. tc05_gemm_kernel<EpTopK> : coarse scores Q^ * P^^T on the tensor cores (tcgen05, TMEM
//      accumulators); the epilogue never stores scores — every thread owns one query row, filters
//      the 128 x BN tile against that query's running threshold and appends survivors to a
//      per-query reservoir that a warp-cooperative radix select compacts to the best k'.
//   3. rescore_kernel : exact scores (fp32 inputs, fp64 accumulate, one rounding to fp32) of the
//      <= n_splits * k' candidates, sort by (score desc, row asc), emit top-k, and CERTIFY: every
//      row that was not a candidate has coarse score <= thr, hence exact score <= thr + eps(q);
//      if thr + eps(q) < k-th exact score the result is provably the exact top-k.
//   4. tier 2, for the queries step 3 could not certify: the SAME coarse kernel once more over those queries only,
//      started from a per-query threshold t(q) = s_k - eps(q) (s_k = k-th exact score found so far, a lower bound of
//      the true one).  Every row that can still belong to the top-k has coarse score > t(q), so unless more than
//      ~2000 rows per split (~4000 / ~8000 above k = 512 / 1024) sit within eps of the boundary nothing is dropped and the result is certified BY
//      CONSTRUCTION: a failed certificate costs one more coarse pass over the failed queries, not a brute force.
//   5. exact_* kernels : what is left (thousands of near-ties at the boundary: duplicated rows, adversarial data) is
//      recomputed by brute force in exact arithmetic.  Also the validation path (ance_index_search_exact).
#include <float.h>
#include <math.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "common.h"
#include "gemm_core.cuh"

namespace {

using namespace tc05;

// Largest k ance_index_search / ance_index_search_exact accept (faiss's GPU flat index has the same limit).
constexpr int kMaxK = 2048;
// Largest k' (candidates kept per split): the default for bf16 operands at k = kMaxK, 2 k + 32.
constexpr int kMaxKprime = 2 * kMaxK + 32;

// ------------------------------------------------------------------------------------------------
// order-preserving float <-> uint32 (larger float -> larger key)
// ------------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint32_t f2ord(float f) {
#ifdef __CUDA_ARCH__
  uint32_t u = __float_as_uint(f);
#else
  uint32_t u;
  memcpy(&u, &f, 4);
#endif
  return u ^ (static_cast<uint32_t>(static_cast<int32_t>(u) >> 31) | 0x80000000u);
}
__host__ __device__ __forceinline__ float ord2f(uint32_t k) {
  uint32_t u = (k & 0x80000000u) ? (k ^ 0x80000000u) : ~k;
#ifdef __CUDA_ARCH__
  return __uint_as_float(u);
#else
  float f;
  memcpy(&f, &u, 4);
  return f;
#endif
}
// 64-bit sort key: score descending, then row ascending  (larger key = better)
__device__ __forceinline__ uint64_t make_key(float score, uint32_t row) {
  return (static_cast<uint64_t>(f2ord(score)) << 32) | static_cast<uint64_t>(0xFFFFFFFFu - row);
}
__device__ __forceinline__ float key_score(uint64_t k) { return ord2f(static_cast<uint32_t>(k >> 32)); }
__device__ __forceinline__ uint32_t key_row(uint64_t k) { return 0xFFFFFFFFu - static_cast<uint32_t>(k); }

template <class T>
__device__ __forceinline__ T* shfl_ptr(T* p, int src) {
  uint64_t v = reinterpret_cast<uint64_t>(p);
  uint32_t lo = __shfl_sync(0xffffffffu, static_cast<uint32_t>(v), src);
  uint32_t hi = __shfl_sync(0xffffffffu, static_cast<uint32_t>(v >> 32), src);
  return reinterpret_cast<T*>((static_cast<uint64_t>(hi) << 32) | lo);
}

// ------------------------------------------------------------------------------------------------
// 1. fp32 -> 16-bit operand rows, with the norms the certificate needs
// ------------------------------------------------------------------------------------------------
// mu (index rows only, may be null): the rows are CENTRED before rounding, x' = x - mu.  <q, x> = <q, x - mu> + <q, mu> and
// the second term is the same for every row, so the ranking is unchanged while every norm in the certificate's error bound
// becomes that of the centred row — embeddings that share a large common component (anisotropic BERT-style outputs, an
// untrained / collapsed encoder) would otherwise spend the 16-bit significand on the component that cannot change the order.
template <bool kBF16>
__global__ void quantize_rows_kernel(const float* __restrict__ X, uint16_t* __restrict__ X16, int64_t n, int d,
                                     const float* __restrict__ mu, float* __restrict__ norm_hat,
                                     float* __restrict__ norm_delta, unsigned int* __restrict__ max_stats,
                                     int* __restrict__ err_flag) {
  // err_flag: set to 1 when a value is non-finite after rounding (fp16 overflow, or inf / NaN in the input)
  const int lane = threadIdx.x & 31;
  const int64_t row = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n) return;
  const float* x = X + row * d;
  uint16_t* o = X16 + row * d;
  float sh = 0.f, sd = 0.f, sx = 0.f;
  bool bad = false;
  for (int i = lane * 4; i < d; i += 128) {  // d % 4 == 0 (checked on the host)
    float4 v = __ldg(reinterpret_cast<const float4*>(x + i));
    if (mu) {
      const float4 m = __ldg(reinterpret_cast<const float4*>(mu + i));
      v.x -= m.x; v.y -= m.y; v.z -= m.z; v.w -= m.w;
    }
    float a[4] = {v.x, v.y, v.z, v.w};
    uint16_t q[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      float back;
      if (kBF16) {
        __nv_bfloat16 h = __float2bfloat16_rn(a[t]);
        q[t] = __bfloat16_as_ushort(h);
        back = __bfloat162float(h);
      } else {
        __half h = __float2half_rn(a[t]);
        q[t] = __half_as_ushort(h);
        back = __half2float(h);
      }
      if (!(fabsf(back) <= 3.0e38f)) bad = true;  // inf / nan after rounding
      sh = fmaf(back, back, sh);
      const float e = a[t] - back;
      sd = fmaf(e, e, sd);
      sx = fmaf(a[t], a[t], sx);
    }
    uint2 pk;
    pk.x = static_cast<uint32_t>(q[0]) | (static_cast<uint32_t>(q[1]) << 16);
    pk.y = static_cast<uint32_t>(q[2]) | (static_cast<uint32_t>(q[3]) << 16);
    *reinterpret_cast<uint2*>(o + i) = pk;
  }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) {
    sh += __shfl_xor_sync(0xffffffffu, sh, s);
    sd += __shfl_xor_sync(0xffffffffu, sd, s);
    sx += __shfl_xor_sync(0xffffffffu, sx, s);
  }
  if (__any_sync(0xffffffffu, bad) && lane == 0 && err_flag) atomicExch(err_flag, 1);
  if (lane == 0) {
    // round the bounds up a little: they are upper bounds in the certificate
    // (the fp32 subtraction x - mu is itself rounded: at most 2^-24 |x - mu| per element, charged to the delta norm)
    const float nh = sqrtf(sh) * 1.00001f, nd = (sqrtf(sd) + (mu ? 1.2e-7f * sqrtf(sx) : 0.f)) * 1.00001f;
    if (norm_hat) norm_hat[row] = nh;
    if (norm_delta) norm_delta[row] = nd;
    if (max_stats) {  // non-negative floats order like their bit patterns
      atomicMax(&max_stats[0], __float_as_uint(nh));
      atomicMax(&max_stats[1], __float_as_uint(nd));
    }
  }
}

// column sums of a slab of rows (fp64), one atomicAdd per (block, column); then mu = sums / n
__global__ void __launch_bounds__(256) column_sum_kernel(const float* __restrict__ X, int64_t n, int d, int slab,
                                                         double* __restrict__ sums) {
  const int64_t r0 = static_cast<int64_t>(blockIdx.x) * slab, r1 = min(n, r0 + slab);
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    double acc = 0.0;
    for (int64_t r = r0; r < r1; ++r) acc += static_cast<double>(__ldg(X + r * d + c));
    atomicAdd(sums + c, acc);
  }
}
__global__ void finalize_mean_kernel(const double* __restrict__ sums, int64_t n, int d, float* __restrict__ mu) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < d) mu[c] = static_cast<float>(sums[c] / static_cast<double>(n));
}

// ------------------------------------------------------------------------------------------------
// 2. coarse pass epilogue: per-query running top-k' over the swept corpus tiles
// ------------------------------------------------------------------------------------------------
template <int BN, int CAP>
struct EpTopK {
  static constexpr uint64_t kHintA = tc05::kEvictLast;   // query tile: re-read for every corpus tile
  static constexpr uint64_t kHintB = tc05::kEvictNormal;  // corpus rows: every concurrently sweeping CTA pair re-reads
                                                          // the same tile from L2 (EVICT_FIRST made each pair go to
                                                          // HBM: 788 GB of DRAM reads for 13.6 GB of operands, ncu r01)
  // CAP <= 2048: the reservoir is selected in registers (kSlots keys and ids per lane).  Larger reservoirs (k > 512) do
  // not fit there: compact_wide selects them where they are, in global memory (L2), with a 256-bin histogram per
  // epilogue warp in shared memory.
  static constexpr bool kWide = CAP > 2048;
  static constexpr int kEpiWarps = 4;
  static constexpr int kSmemBytes = kWide ? kEpiWarps * 256 * 4 : 0;
  struct Params {
    float* scratch_sc;  // [gridDim.x * 128 * CAP] reservoir scores
    int* scratch_id;    // [gridDim.x * 128 * CAP] reservoir rows
    int* cand_id;       // [nq * n_splits * out_cap]
    int* cand_cnt;      // [nq * n_splits]
    float* cand_thr;    // [nq * n_splits]  final running threshold: every row NOT in the candidate list has coarse score <= it
    const float* thr_init;  // [nq] starting threshold per query (tier 2), or null: -inf
    int kprime;         // a reservoir that fills up is compacted to its best kprime entries
    int out_cap;        // entries kept per (query, split) at the end: kprime (tier 1) or the reservoir size (tier 2: nothing
                        // that passed the threshold is dropped unless the reservoir itself overflowed)
    int nq, n_rows;
  };

  float thr;
  int cnt;
  float* sc;
  int* id;

  __device__ __forceinline__ void begin_work(const Params& p, const gemm::WorkShape&, const gemm::EpiCtx& cx) {
    const int r = cx.quad * 32 + cx.lane;
    const size_t base = (static_cast<size_t>(blockIdx.x) * gemm::BM + r) * CAP;
    sc = p.scratch_sc + base;
    id = p.scratch_id + base;
    thr = (cx.row0 + r < p.nq) ? (p.thr_init ? __ldg(p.thr_init + cx.row0 + r) : -INFINITY) : INFINITY;
    cnt = 0;
  }

  // Warp-cooperative exact selection of the best kprime entries of lane `src`'s reservoir
  // (radix select on the order-preserving key, stable compaction: among equal scores the earlier
  // = lower row wins).  Afterwards src.cnt = kprime and src.thr = kprime-th best coarse score.
  __device__ __forceinline__ void compact(int kprime, int src, int lane) {
    constexpr int kSlots = CAP / 32;
    const int n = __shfl_sync(0xffffffffu, cnt, src);
    float* s_sc = shfl_ptr(sc, src);
    int* s_id = shfl_ptr(id, src);
    uint32_t keys[kSlots];
    int ids[kSlots];
#pragma unroll
    for (int j = 0; j < kSlots; ++j) {
      const int i = j * 32 + lane;
      const bool v = i < n;
      keys[j] = v ? f2ord(s_sc[i]) : 0u;
      ids[j] = v ? s_id[i] : -1;
    }
    uint32_t prefix = 0;
    int remaining = kprime;
#pragma unroll 1
    for (int b = 31; b >= 0; --b) {
      const uint32_t cand = prefix | (1u << b);
      const uint32_t mask = ~((1u << b) - 1u);
      int c = 0;
#pragma unroll
      for (int j = 0; j < kSlots; ++j) c += ((keys[j] & mask) == cand) ? 1 : 0;
      c = __reduce_add_sync(0xffffffffu, c);
      if (c >= remaining) prefix = cand;
      else remaining -= c;
    }
    const uint32_t T = prefix;
    const unsigned lt = (1u << lane) - 1u;
    int base = 0, eq_seen = 0;
#pragma unroll
    for (int j = 0; j < kSlots; ++j) {
      const bool gt = keys[j] > T, eq = keys[j] == T;
      const unsigned eqm = __ballot_sync(0xffffffffu, eq);
      const bool keep = gt || (eq && (eq_seen + __popc(eqm & lt)) < remaining);
      const unsigned km = __ballot_sync(0xffffffffu, keep);
      if (keep) {
        const int pos = base + __popc(km & lt);
        s_sc[pos] = ord2f(keys[j]);
        s_id[pos] = ids[j];
      }
      base += __popc(km);
      eq_seen += __popc(eqm);
    }
    __syncwarp();
    if (lane == src) {
      cnt = kprime;
      thr = ord2f(T);
    }
  }

  // Same selection and the same result as compact() for a reservoir too large for registers: four passes of an
  // 8-bit-digit radix select (most significant digit first) over the reservoir in place, each counting the entries
  // that match the digits chosen so far into the warp's shared histogram, then the same stable in-place compaction.
  // Every dropped entry has key < T, or key == T behind the `remaining` kept ones: coarse score <= thr, as the
  // certificate requires.
  __device__ __forceinline__ void compact_wide(int kprime, int src, int lane, uint32_t* hist) {
    const int n = __shfl_sync(0xffffffffu, cnt, src);
    float* s_sc = shfl_ptr(sc, src);
    int* s_id = shfl_ptr(id, src);
    uint32_t prefix = 0, pmask = 0;
    int remaining = kprime;   // n > kprime: entries matching the prefix always number >= remaining
#pragma unroll 1
    for (int shift = 24; shift >= 0; shift -= 8) {
      for (int b = lane; b < 256; b += 32) hist[b] = 0u;
      __syncwarp();
      for (int i0 = 0; i0 < n; i0 += 32) {
        // lanes whose entries share a digit add once for all of them: in the first passes most entries fall in a few
        // bins, and 32 atomics on one shared-memory address serialise
        const int i = i0 + lane;
        uint32_t bin = 256u;   // no entry, or one that does not match the digits chosen so far
        if (i < n) {
          const uint32_t key = f2ord(s_sc[i]);
          if ((key & pmask) == prefix) bin = (key >> shift) & 255u;
        }
        const unsigned peers = __match_any_sync(0xffffffffu, bin);
        if (bin < 256u && lane == __ffs(peers) - 1) atomicAdd(&hist[bin], static_cast<uint32_t>(__popc(peers)));
      }
      __syncwarp();
      // lane l owns digits 8l .. 8l+7; `above` = entries whose digit belongs to a higher lane
      int c[8], tot = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        c[j] = static_cast<int>(hist[lane * 8 + j]);
        tot += c[j];
      }
      int suf = tot;
#pragma unroll
      for (int s = 1; s < 32; s <<= 1) {
        const int v = __shfl_down_sync(0xffffffffu, suf, s);
        if (lane + s < 32) suf += v;
      }
      const int above = suf - tot;
      const bool mine = above < remaining && remaining <= suf;   // exactly one lane
      int digit = 0, rem = 0;
      if (mine) {
        int acc = above;
#pragma unroll
        for (int j = 7; j >= 0; --j) {
          if (acc + c[j] >= remaining) {
            digit = lane * 8 + j;
            rem = remaining - acc;
            break;
          }
          acc += c[j];
        }
      }
      const int owner = __ffs(__ballot_sync(0xffffffffu, mine)) - 1;
      digit = __shfl_sync(0xffffffffu, digit, owner);
      remaining = __shfl_sync(0xffffffffu, rem, owner);
      prefix |= static_cast<uint32_t>(digit) << shift;
      pmask |= 255u << shift;
    }
    const uint32_t T = prefix;
    const unsigned lt = (1u << lane) - 1u;
    int base = 0, eq_seen = 0;
#pragma unroll 1
    for (int i0 = 0; i0 < n; i0 += 32) {
      const int i = i0 + lane;
      const bool v = i < n;
      const float s = v ? s_sc[i] : 0.f;
      const int rid = v ? s_id[i] : -1;
      const uint32_t key = f2ord(s);
      const bool gt = v && key > T, eq = v && key == T;
      const unsigned eqm = __ballot_sync(0xffffffffu, eq);
      const bool keep = gt || (eq && (eq_seen + __popc(eqm & lt)) < remaining);
      const unsigned km = __ballot_sync(0xffffffffu, keep);
      __syncwarp();   // every lane has read its entry of this chunk before any lane overwrites one (pos <= i0 + 31)
      if (keep) {
        const int pos = base + __popc(km & lt);
        s_sc[pos] = s;
        s_id[pos] = rid;
      }
      base += __popc(km);
      eq_seen += __popc(eqm);
    }
    __syncwarp();
    if (lane == src) {
      cnt = kprime;
      thr = ord2f(T);
    }
  }

  __device__ __forceinline__ void compact_any(int kprime, int src, const gemm::EpiCtx& cx) {
    if constexpr (kWide) compact_wide(kprime, src, cx.lane, reinterpret_cast<uint32_t*>(cx.ep_smem) + cx.epi_warp * 256);
    else compact(kprime, src, cx.lane);
  }

  __device__ __forceinline__ void tile(const Params& p, const gemm::WorkShape&, const gemm::EpiCtx& cx,
                                       uint32_t tacc, int nb) {
#pragma unroll 1
    for (int c = 0; c < BN; c += 32) {
      uint32_t v[32];
      tmem_ld_32x32b_x32(tacc + c, v);
      tmem_ld_wait();
      float m = __uint_as_float(v[0]);
#pragma unroll
      for (int i = 1; i < 32; ++i) m = fmaxf(m, __uint_as_float(v[i]));
      if (m > thr) {
        const int col0 = nb * BN + c;
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const float s = __uint_as_float(v[i]);
          if (s > thr && col0 + i < p.n_rows) {  // rows past the end are TMA zero fill
            sc[cnt] = s;
            id[cnt] = col0 + i;
            ++cnt;
          }
        }
      }
      __syncwarp();
      unsigned need = __ballot_sync(0xffffffffu, cnt > CAP - 32);
      while (need) {
        const int src = __ffs(need) - 1;
        need &= need - 1;
        compact_any(p.kprime, src, cx);
      }
    }
  }

  __device__ __forceinline__ void end_kernel(const Params&, const gemm::EpiCtx&) {}

  __device__ __forceinline__ void end_work(const Params& p, const gemm::WorkShape& ws, const gemm::EpiCtx& cx) {
    __syncwarp();
    unsigned need = __ballot_sync(0xffffffffu, cnt > p.out_cap);
    while (need) {
      const int src = __ffs(need) - 1;
      need &= need - 1;
      compact_any(p.kprime, src, cx);
    }
    for (int l = 0; l < 32; ++l) {
      const int row = cx.row0 + cx.quad * 32 + l;
      if (row >= p.nq) break;  // warp-uniform
      const int n = __shfl_sync(0xffffffffu, cnt, l);
      const float t = __shfl_sync(0xffffffffu, thr, l);
      const int* s_id = shfl_ptr(id, l);
      const size_t slot = static_cast<size_t>(row) * ws.n_splits + cx.split;
      int* out = p.cand_id + slot * p.out_cap;
      for (int i = cx.lane; i < n; i += 32) out[i] = s_id[i];
      if (cx.lane == 0) {
        p.cand_cnt[slot] = n;
        p.cand_thr[slot] = t;
      }
    }
    __syncwarp();
  }
};

// ------------------------------------------------------------------------------------------------
// shared helpers: exact dot products and block bitonic sort
// ------------------------------------------------------------------------------------------------
// exact <q, p>: fp32 inputs, products and sum in fp64 (each product is exact in fp64), result
// rounded once to fp32.  Lane-strided float4 loads; deterministic shuffle tree.
__device__ __forceinline__ double warp_dot_f64(const float* __restrict__ q_smem, const float* __restrict__ p, int d,
                                               int lane) {
  double acc = 0.0;
  if ((d & 127) == 0) {
    for (int i = lane * 4; i < d; i += 128) {
      const float4 a = *reinterpret_cast<const float4*>(q_smem + i);
      const float4 b = __ldg(reinterpret_cast<const float4*>(p + i));
      acc = fma(static_cast<double>(a.x), static_cast<double>(b.x), acc);
      acc = fma(static_cast<double>(a.y), static_cast<double>(b.y), acc);
      acc = fma(static_cast<double>(a.z), static_cast<double>(b.z), acc);
      acc = fma(static_cast<double>(a.w), static_cast<double>(b.w), acc);
    }
  } else {
    for (int i = lane; i < d; i += 32) acc = fma(static_cast<double>(q_smem[i]), static_cast<double>(__ldg(p + i)), acc);
  }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
  return acc;
}

// descending bitonic sort of n (power of two) 64-bit keys in shared memory by the whole block
__device__ __forceinline__ void block_bitonic_desc(uint64_t* keys, int n) {
  for (int size = 2; size <= n; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      __syncthreads();
      for (int t = threadIdx.x; t < (n >> 1); t += blockDim.x) {
        const int lo = 2 * t - (t & (stride - 1));
        const int hi = lo + stride;
        const bool desc = ((lo & size) == 0);
        const uint64_t a = keys[lo], b = keys[hi];
        if ((a < b) == desc) {
          keys[lo] = b;
          keys[hi] = a;
        }
      }
    }
  }
  __syncthreads();
}

__host__ __device__ inline int next_pow2(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

// ------------------------------------------------------------------------------------------------
// 3. exact rescoring of the candidates + certificate
// ------------------------------------------------------------------------------------------------
struct RescoreParams {
  const float* Q;
  const float* P;
  int d;
  const int* cand_id;
  const int* cand_cnt;
  const float* cand_thr;
  int n_splits, cand_stride, k;   // cand_stride = EpTopK out_cap
  const float* qn_hat;
  const float* qn_delta;
  const unsigned int* pstats;  // [0] max ||p^||, [1] max ||p - p^|| (float bits) of the CENTRED rows
  const float* mu;             // the centre subtracted from every index row before rounding (null: none)
  float accum_rel;             // bound on the tensor core's accumulation error / (||q^|| ||p^||), see coarse_rescore_pass
  float* D;
  int64_t* I;
  int64_t row_offset;
  const int* qlist;    // block b handles candidate slot b of query qlist[b] (null: query b)
  int* flagged_list;   // uncertified queries of this pass
  float* flagged_thr;  // starting threshold of the next tier for flagged_list[i] (null: not needed)
  int flag_slot;       // counters[flag_slot] counts them
  int* counters;       // [0] tier-1 flagged [1] n_candidates [2] max eps bits [3] tier-2 flagged
  unsigned int* max_eps;
  int sort_n;          // pow2 >= total candidates of a query
};

// exact <q, p_c> of kNB candidate rows at once: all the row's 16-byte loads (d / 128 per lane and row) are issued
// before the first fp64 FMA, so a warp keeps kNB * d / 128 gathers in flight instead of one (the rows are random
// 3 KB reads: latency, not bandwidth, bounded the one-row-at-a-time form at 0.14 of HBM).  kJ = d / 128 (768: kJ = 6).
template <int kNB, int kJ>
__device__ __forceinline__ void warp_dots_f64(const float* __restrict__ q_smem, const float* const (&rows)[kNB], int d,
                                              int lane, double (&out)[kNB]) {
  float4 b[kNB][kJ];
#pragma unroll
  for (int j = 0; j < kJ; ++j) {
    {
#pragma unroll
      for (int c = 0; c < kNB; ++c) b[c][j] = __ldg(reinterpret_cast<const float4*>(rows[c] + j * 128 + lane * 4));
    }
  }
#pragma unroll
  for (int c = 0; c < kNB; ++c) out[c] = 0.0;
#pragma unroll
  for (int j = 0; j < kJ; ++j) {
    {
      const float4 a = *reinterpret_cast<const float4*>(q_smem + j * 128 + lane * 4);
#pragma unroll
      for (int c = 0; c < kNB; ++c) {   // same association as warp_dot_f64: the result is bit-identical
        out[c] = fma(static_cast<double>(a.x), static_cast<double>(b[c][j].x), out[c]);
        out[c] = fma(static_cast<double>(a.y), static_cast<double>(b[c][j].y), out[c]);
        out[c] = fma(static_cast<double>(a.z), static_cast<double>(b[c][j].z), out[c]);
        out[c] = fma(static_cast<double>(a.w), static_cast<double>(b[c][j].w), out[c]);
      }
    }
  }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) {
#pragma unroll
    for (int c = 0; c < kNB; ++c) out[c] += __shfl_xor_sync(0xffffffffu, out[c], s);
  }
}

__global__ void __launch_bounds__(256) rescore_kernel(const RescoreParams p) {
  extern __shared__ __align__(16) uint8_t rs_smem[];
  uint64_t* keys = reinterpret_cast<uint64_t*>(rs_smem);
  float* qs = reinterpret_cast<float*>(keys + p.sort_n);
  int* offs = reinterpret_cast<int*>(qs + p.d);  // [n_splits + 1]
  const int ql = blockIdx.x;                       // slot in the candidate arrays
  const int q = p.qlist ? p.qlist[ql] : ql;        // query number (rows of Q, D, I)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;

  for (int i = threadIdx.x; i < p.d; i += blockDim.x) qs[i] = p.Q[static_cast<size_t>(q) * p.d + i];
  if (threadIdx.x == 0) {
    int o = 0;
    for (int s = 0; s < p.n_splits; ++s) {
      offs[s] = o;
      o += p.cand_cnt[static_cast<size_t>(ql) * p.n_splits + s];
    }
    offs[p.n_splits] = o;
  }
  __syncthreads();
  const int m = offs[p.n_splits];
  for (int i = threadIdx.x; i < p.sort_n; i += blockDim.x) keys[i] = 0ull;
  // <q, mu> in fp64: what separates the coarse (centred) scores from the exact ones, identically for every row
  __shared__ double s_qmu[8];
  {
    double part = 0.0;
    if (p.mu)
      for (int i = threadIdx.x; i < p.d; i += blockDim.x) part = fma(static_cast<double>(qs[i]), static_cast<double>(__ldg(p.mu + i)), part);
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) part += __shfl_xor_sync(0xffffffffu, part, s);
    if (lane == 0) s_qmu[warp] = part;
  }
  __syncthreads();
  constexpr int kNB = 4;
  const bool wide = p.d == 768;   // the path's dimension (models.py:145-146); other dims take the one-row loop
  for (int s = 0; s < p.n_splits; ++s) {
    const int n = offs[s + 1] - offs[s];
    const int* ids = p.cand_id + (static_cast<size_t>(ql) * p.n_splits + s) * p.cand_stride;
    if (wide) {
      for (int c0 = warp * kNB; c0 < n; c0 += nwarps * kNB) {
        int row[kNB];
        const float* rp[kNB];
#pragma unroll
        for (int c = 0; c < kNB; ++c) {
          row[c] = ids[min(c0 + c, n - 1)];
          rp[c] = p.P + static_cast<size_t>(row[c]) * p.d;
        }
        double dot[kNB];
        warp_dots_f64<kNB, 6>(qs, rp, p.d, lane, dot);
        if (lane == 0) {
#pragma unroll
          for (int c = 0; c < kNB; ++c)
            if (c0 + c < n) keys[offs[s] + c0 + c] = make_key(static_cast<float>(dot[c]), static_cast<uint32_t>(row[c]));
        }
      }
    } else {
      for (int c = warp; c < n; c += nwarps) {
        const int row = ids[c];
        const double dot = warp_dot_f64(qs, p.P + static_cast<size_t>(row) * p.d, p.d, lane);
        if (lane == 0) keys[offs[s] + c] = make_key(static_cast<float>(dot), static_cast<uint32_t>(row));
      }
    }
  }
  block_bitonic_desc(keys, p.sort_n);
  for (int i = threadIdx.x; i < p.k; i += blockDim.x) {
    const bool ok = i < m;
    p.D[static_cast<size_t>(q) * p.k + i] = ok ? key_score(keys[i]) : -FLT_MAX;
    p.I[static_cast<size_t>(q) * p.k + i] = ok ? p.row_offset + static_cast<int64_t>(key_row(keys[i])) : -1;
  }
  if (threadIdx.x == 0) {
    float thr = -INFINITY;
    for (int s = 0; s < p.n_splits; ++s) thr = fmaxf(thr, p.cand_thr[static_cast<size_t>(ql) * p.n_splits + s]);
    const float maxp = __uint_as_float(p.pstats[0]), maxdp = __uint_as_float(p.pstats[1]);
    const float qn = p.qn_hat[q], qd = p.qn_delta[q];
    // |coarse_j - <q, p_j>| <= eps for EVERY row j (Cauchy-Schwarz on the operand rounding + the accumulation bound);
    // the factor covers the fp32 roundings of this expression itself (norms are already rounded up)
    const float eps = (qd * maxp + qn * maxdp + qd * maxdp + p.accum_rel * qn * maxp) * 1.0001f;
    // A row that is not a candidate has centred coarse score <= thr, hence exact score <= thr + eps + <q, mu>.  The k-th
    // exact score is an fp64 dot product rounded to fp32: the unrounded value is >= sk_lo.  Compared in fp64.
    double qmu = 0.0;
    for (int w2 = 0; w2 < nwarps; ++w2) qmu += s_qmu[w2];
    const double qmu_up = qmu + fabs(qmu) * 1.0e-12;
    const double sk = (m >= p.k) ? static_cast<double>(key_score(keys[p.k - 1])) : -INFINITY;
    const double sk_lo = sk - fabs(sk) * 1.2e-7;
    bool certified;
    if (thr == -INFINITY) certified = true;       // every row of the index was a candidate
    else if (m < p.k) certified = false;          // cannot happen (thr finite => >= k candidates passed it)
    else certified = (static_cast<double>(thr) + static_cast<double>(eps) + qmu_up < sk_lo);
    atomicAdd(&p.counters[1], m);
    atomicMax(p.max_eps, __float_as_uint(eps));
    if (!certified) {
      const int slot = atomicAdd(&p.counters[p.flag_slot], 1);
      p.flagged_list[slot] = q;
      if (p.flagged_thr) {
        // Next tier starts from t < s_k - eps: every row whose exact score reaches s_k (the k-th exact score found so
        // far, a lower bound of the final one) has coarse score >= s_k - eps > t, i.e. passes the filter.
        const float x = __double2float_rd(sk_lo - qmu_up - static_cast<double>(eps));   // in centred coarse-score units
        p.flagged_thr[slot] = (m < p.k) ? -INFINITY : __fsub_rd(x, fmaxf(fabsf(x), eps) * 1.0e-6f);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// 4. exact brute force (fallback for uncertified queries, and the validation path)
// ------------------------------------------------------------------------------------------------
constexpr int kExQB = 4;       // queries per block
constexpr int kExRound = 16;   // rows per warp between reservoir checks
constexpr int kExWarps = 8;    // 256 threads
// reservoir keys per query (kExBuf, a template argument): a compacted reservoir holds k keys and takes up to
// kExWarps * kExRound more before the next check, so at least k + kExWarps * kExRound; and at least 2 k, so that a
// compaction (a block-wide sort) is paid for by about k new keys, not by one round's.  A power of two: 1024 for every
// k <= 512, 2048 up to k = 1024, 4096 up to k = 2048.
__host__ __device__ constexpr int exact_buf_keys(int k) {
  int b = 1024;
  while (b < k + kExWarps * kExRound || b < 2 * k) b <<= 1;
  return b;
}

struct ExactParams {
  const float* Q;
  const float* P;
  int d;
  int64_t n_rows;
  const int* qlist;      // query numbers (null = q_base + i)
  int q_base;
  const int* nq_dev;     // number of queries on the device (null = use nq)
  int nq;
  int k;                 // <= kMaxK
  int n_chunks;
  uint64_t* chunk_keys;  // [nq_cap * n_chunks * k]
};

template <int kExBuf>
__global__ void __launch_bounds__(256) exact_chunk_kernel(const ExactParams p) {
  extern __shared__ __align__(16) uint8_t ex_smem[];
  uint64_t* buf = reinterpret_cast<uint64_t*>(ex_smem);              // [kExQB][kExBuf]
  float* qs = reinterpret_cast<float*>(buf + kExQB * kExBuf);        // [kExQB][d]
  __shared__ int cnt[kExQB];
  __shared__ unsigned long long thr[kExQB];
  const int nq = p.nq_dev ? min(*p.nq_dev, p.nq) : p.nq;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int64_t rows_per_chunk = (p.n_rows + p.n_chunks - 1) / p.n_chunks;
  const int64_t r0 = static_cast<int64_t>(blockIdx.x) * rows_per_chunk;
  const int64_t r1 = min(p.n_rows, r0 + rows_per_chunk);

  for (int g = blockIdx.y; g * kExQB < nq; g += gridDim.y) {
    const int nqb = min(kExQB, nq - g * kExQB);
    __syncthreads();
    for (int i = threadIdx.x; i < kExQB * p.d; i += blockDim.x) {
      const int qi = i / p.d, e = i - qi * p.d;
      float v = 0.f;
      if (qi < nqb) {
        const int q = p.qlist ? p.qlist[g * kExQB + qi] : p.q_base + g * kExQB + qi;
        v = p.Q[static_cast<size_t>(q) * p.d + e];
      }
      qs[i] = v;
    }
    if (threadIdx.x < kExQB) {
      cnt[threadIdx.x] = 0;
      thr[threadIdx.x] = 0ull;
    }
    __syncthreads();
    for (int64_t base = r0; base < r1; base += static_cast<int64_t>(nwarps) * kExRound) {
      for (int t = 0; t < kExRound; ++t) {
        const int64_t row = base + static_cast<int64_t>(t) * nwarps + warp;
        if (row >= r1) break;
        const float* prow = p.P + row * p.d;
        double acc[kExQB];
#pragma unroll
        for (int qi = 0; qi < kExQB; ++qi) acc[qi] = 0.0;
        for (int i = lane; i < p.d; i += 32) {
          const double b = static_cast<double>(__ldg(prow + i));
#pragma unroll
          for (int qi = 0; qi < kExQB; ++qi) acc[qi] = fma(static_cast<double>(qs[qi * p.d + i]), b, acc[qi]);
        }
#pragma unroll
        for (int qi = 0; qi < kExQB; ++qi) {
#pragma unroll
          for (int s = 16; s > 0; s >>= 1) acc[qi] += __shfl_xor_sync(0xffffffffu, acc[qi], s);
        }
        if (lane < nqb) {
          double a = acc[0];
#pragma unroll
          for (int qi = 1; qi < kExQB; ++qi)
            if (lane == qi) a = acc[qi];
          const uint64_t key = make_key(static_cast<float>(a), static_cast<uint32_t>(row));
          if (key > thr[lane]) {
            const int slot = atomicAdd(&cnt[lane], 1);
            buf[lane * kExBuf + slot] = key;  // slot < kExBuf: at most nwarps*kExRound appends per round
          }
        }
      }
      __syncthreads();
      for (int qi = 0; qi < nqb; ++qi) {
        if (cnt[qi] > kExBuf - nwarps * kExRound) {  // block-uniform
          const int n = cnt[qi];
          for (int i = n + threadIdx.x; i < kExBuf; i += blockDim.x) buf[qi * kExBuf + i] = 0ull;
          block_bitonic_desc(buf + qi * kExBuf, kExBuf);
          if (threadIdx.x == 0) {
            cnt[qi] = p.k;
            thr[qi] = buf[qi * kExBuf + p.k - 1];
          }
          __syncthreads();
        }
      }
    }
    __syncthreads();
    for (int qi = 0; qi < nqb; ++qi) {
      const int n = cnt[qi];
      for (int i = n + threadIdx.x; i < kExBuf; i += blockDim.x) buf[qi * kExBuf + i] = 0ull;
      block_bitonic_desc(buf + qi * kExBuf, kExBuf);
      uint64_t* out = p.chunk_keys + (static_cast<size_t>(g * kExQB + qi) * p.n_chunks + blockIdx.x) * p.k;
      for (int i = threadIdx.x; i < p.k; i += blockDim.x) out[i] = (i < n) ? buf[qi * kExBuf + i] : 0ull;
    }
  }
}

constexpr int kMergeBuf = 4096;
static_assert(kMergeBuf >= 2 * kMaxK, "exact_merge_kernel takes kMergeBuf - k new keys per round");

__global__ void __launch_bounds__(256) exact_merge_kernel(const ExactParams p, float* D, int64_t* I, int out_k,
                                                          int64_t row_offset) {
  __shared__ uint64_t keys[kMergeBuf];
  const int nq = p.nq_dev ? min(*p.nq_dev, p.nq) : p.nq;
  for (int qi = blockIdx.x; qi < nq; qi += gridDim.x) {
    const int q = p.qlist ? p.qlist[qi] : p.q_base + qi;
    const uint64_t* src = p.chunk_keys + static_cast<size_t>(qi) * p.n_chunks * p.k;
    const int total = p.n_chunks * p.k;
    int have = 0;  // keys[0..have) = current best (sorted)
    int pos = 0;
    __syncthreads();
    while (pos < total) {
      const int take = min(kMergeBuf - have, total - pos);
      for (int i = threadIdx.x; i < take; i += blockDim.x) keys[have + i] = src[pos + i];
      for (int i = have + take + threadIdx.x; i < kMergeBuf; i += blockDim.x) keys[i] = 0ull;
      pos += take;
      block_bitonic_desc(keys, kMergeBuf);
      have = p.k;
    }
    for (int i = threadIdx.x; i < out_k; i += blockDim.x) {
      const uint64_t key = (i < p.k) ? keys[i] : 0ull;
      const bool ok = key != 0ull;
      D[static_cast<size_t>(q) * out_k + i] = ok ? key_score(key) : -FLT_MAX;
      I[static_cast<size_t>(q) * out_k + i] = ok ? row_offset + static_cast<int64_t>(key_row(key)) : -1;
    }
    __syncthreads();
  }
}

// 16-bit operand rows of the listed queries -> compact matrix (second, wider coarse pass)
__global__ void gather_rows16_kernel(const uint16_t* __restrict__ src, const int* __restrict__ qlist, int n, int d,
                                     uint16_t* __restrict__ dst) {
  const int r = blockIdx.x;
  if (r >= n) return;
  const uint4* s = reinterpret_cast<const uint4*>(src + static_cast<size_t>(qlist[r]) * d);
  uint4* o = reinterpret_cast<uint4*>(dst + static_cast<size_t>(r) * d);
  for (int i = threadIdx.x; i < d / 8; i += blockDim.x) o[i] = s[i];
}

}  // namespace

// ================================================================================================
// index handle
// ================================================================================================
struct ance_index {
  int dim = 0;
  int64_t cap = 0, n = 0;
  int fmt = ANCE_FMT_FP16;
  int device = 0;
  float* P32 = nullptr;      // [cap, dim]
  bool owns_p32 = true;      // false: caller-owned storage (ance_index_create_over)
  uint16_t* P16 = nullptr;   // [cap, dim]
  unsigned int* pstats = nullptr;  // [2]
  float* mu = nullptr;             // [dim] centre of the rows (see quantize_rows_kernel)
  double* colsum = nullptr;        // [dim]
  bool dirty = false;              // rows were added / the format changed since the 16-bit operands were (re)built
  bool centred = false;
  int center = 1;                  // tunable "center": subtract the column mean before rounding
  // tunables
  int kprime = 0, n_splits = 0, cta_group = 2, max_ctas = 0, exact_fallback = 1, tier2 = 1, pace_window = 16;
  // workspace (grown lazily)
  uint16_t* Q16 = nullptr; float* qn_hat = nullptr; float* qn_delta = nullptr; int64_t q_cap = 0;
  float* scratch_sc = nullptr; int* scratch_id = nullptr; size_t scratch_elems = 0;
  int* cand_id = nullptr; int* cand_cnt = nullptr; float* cand_thr = nullptr; size_t cand_slots = 0, cand_ids = 0;
  int* flagged = nullptr; float* flagged_thr = nullptr; int64_t flagged_cap = 0;
  int* flagged2 = nullptr; size_t flagged2_cap = 0;
  uint16_t* Q16b = nullptr; size_t q16b_elems = 0;
  int* pace = nullptr;              // [kMaxPace] progress counters of the sweeping CTA pairs (soft barrier)
  // [0] tier-1 flagged  [1] candidates rescored  [2] max eps bits  [3] tier-2 flagged  [4,5] spare
  // [6] a QUERY was non-finite after rounding (cleared per search)  [7] an index ROW was (sticky until reset / requantise)
  int* counters = nullptr;
  uint64_t* chunk_keys = nullptr; size_t chunk_keys_elems = 0;
  // last search
  ance_search_stats stats{};
  cudaStream_t last_stream = nullptr;
};

namespace {

constexpr int kMaxPace = 256;
constexpr int kCntQueryErr = 6, kCntRowErr = 7, kNumCounters = 8;

template <class T>
int ensure(T** ptr, size_t* have, size_t want) {
  if (*have >= want) return ANCE_OK;
  if (*ptr) cudaFree(*ptr);
  *ptr = nullptr;
  *have = 0;
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(ptr), want * sizeof(T));
  if (e != cudaSuccess) {
    ance::set_error("cudaMalloc(%zu bytes) failed: %s", want * sizeof(T), cudaGetErrorString(e));
    return ANCE_ERR_NOMEM;
  }
  *have = want;
  return ANCE_OK;
}

int check_device() {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) {
    ance::set_error("no CUDA device: %s (libance_b200 has no CPU fallback)", cudaGetErrorString(e));
    return ANCE_ERR_CUDA;
  }
  int major = 0;
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (major != 10) {
    ance::set_error("device %d has compute capability %d.x; libance_b200 is built for sm_100a only", dev, major);
    return ANCE_ERR_CUDA;
  }
  return ANCE_OK;
}

// handles are bound to the device that was current at creation (header): refuse anything else instead of launching
// on the wrong GPU
int check_handle_device(const ance_index* ix, const char* who) {
  int dev = -1;
  ANCE_CUDA(cudaGetDevice(&dev));
  ANCE_REQUIRE(dev == ix->device, "%s: the index belongs to device %d but device %d is current", who, ix->device, dev);
  return ANCE_OK;
}

// Reservoir entries per query row of the coarse epilogue for a given k': room for about k' more survivors between two
// compactions.  k <= 512 only ever uses 1024 and 2048 (k' <= 992).
int reservoir_cap(int kprime) { return kprime <= 512 ? 1024 : kprime <= 1024 ? 2048 : kprime <= 2048 ? 4096 : 8192; }

// Candidates per query above k = 512, all splits together: the rescore's shared-memory sort, 16384 keys = 128 KB.
constexpr int kMaxCands = 16384;
static_assert(kMaxKprime <= kMaxCands, "one split's candidates must fit the rescore's sort");

// k' of tier 2 (its reservoir is compacted only when it overflows, dropping candidates): half a reservoir less one
// compaction check — CAP 2048 for k <= 512 (as it always was), 4096 up to k = 1024, 8192 up to kMaxK.
int tier2_kprime(int k) { return k <= 512 ? 992 : k <= 1024 ? 2016 : 4064; }

template <int BN, int STAGES, int CG, int CAP, uint32_t FMT>
int launch_coarse(ance_index* ix, const uint16_t* Q16, int64_t nq, int kprime, int out_cap, const float* thr_init,
                  int n_splits_req, int* n_splits_out, cudaStream_t st) {
  using Ep = EpTopK<BN, CAP>;
  const int N = static_cast<int>(ix->n);
  gemm::WorkShape ws = gemm::make_shape(static_cast<int>(nq), N, ix->dim, BN, CG, n_splits_req);
  *n_splits_out = ws.n_splits;
  // One sweep per query tile: every concurrently running CTA pair re-reads the same corpus tile, so keep it in L2.
  // With row-range splits each pair streams its own range once: do not let it evict the (re-read) query tiles.
  ws.hint_b = (ws.n_splits == 1) ? tc05::kEvictNormal : tc05::kEvictFirst;
  CUtensorMap tmA, tmB;
  if (!tc05_host::make_tmap_2d_16b(&tmA, Q16, nq, ix->dim, ix->dim, gemm::BM) ||
      !tc05_host::make_tmap_2d_16b(&tmB, ix->P16, ix->n, ix->dim, ix->dim, BN / CG)) {
    ance::set_error("cuTensorMapEncodeTiled failed (nq=%lld n=%lld d=%d)", (long long)nq, (long long)ix->n, ix->dim);
    return ANCE_ERR_CUDA;
  }
  const int ctas = (ix->max_ctas > 0 ? ix->max_ctas : gemm::sm_count());
  // one reservoir of max(CAP, 2048) entries per (CTA, query row): the large-k reservoirs (CAP 8192: 1.2 GB on 148 SMs)
  // are allocated only when a large k is searched
  const size_t res = static_cast<size_t>(ctas) * gemm::BM * std::max(CAP, 2048);
  size_t se = ix->scratch_elems;
  int rc = ensure(&ix->scratch_sc, &se, res);
  if (rc) return rc;
  se = ix->scratch_elems;
  rc = ensure(&ix->scratch_id, &se, res);
  if (rc) return rc;
  ix->scratch_elems = se;
  const size_t slots = static_cast<size_t>(nq) * ws.n_splits;
  size_t a = ix->cand_slots, b = ix->cand_slots;
  if ((rc = ensure(&ix->cand_cnt, &a, slots))) return rc;
  if ((rc = ensure(&ix->cand_thr, &b, slots))) return rc;
  ix->cand_slots = a;
  if ((rc = ensure(&ix->cand_id, &ix->cand_ids, slots * out_cap))) return rc;
  // Soft barrier between the sweeping CTA pairs (gemm_core.cuh): pairs that sweep the SAME corpus rows share each tile
  // through L2 as long as they stay within `pace_window` tiles of each other.  Without it they drift apart and every one of
  // them streams the rows from HBM by itself (ncu, round 1: 788 GB of DRAM reads for a 13.6 GB operand; measured round 2 at
  // 18,944 and 75,776 queries: 910 -> 1213 TFLOP/s with the barrier).  Two shapes qualify: every item sweeps the whole
  // corpus (n_splits == 1: all pairs pace each other), or one wave of (query tile, row range) items (pairs with the same
  // range pace each other).
  const int total_items = ws.num_m_blks * ws.n_splits;
  const int clusters = std::min(total_items, ctas / CG);
  const bool whole = ws.n_splits == 1 && clusters > 1;
  const bool one_wave = ws.n_splits > 1 && ws.num_m_blks > 1 && total_items <= ctas / CG;
  if ((whole || one_wave) && clusters <= kMaxPace && ix->pace_window > 0 && ws.n_blks_per_split > 4 * ix->pace_window) {
    ANCE_CUDA(cudaMemsetAsync(ix->pace, 0, kMaxPace * sizeof(int), st));
    ws.pace = ix->pace;
    ws.pace_window = ix->pace_window;
    ws.pace_stride = whole ? 1 : ws.n_splits;
    ws.hint_b = tc05::kEvictNormal;   // the tile is re-read by the other pairs of the group: keep it in L2
  }
  typename Ep::Params p;
  p.scratch_sc = ix->scratch_sc;
  p.scratch_id = ix->scratch_id;
  p.cand_id = ix->cand_id;
  p.cand_cnt = ix->cand_cnt;
  p.cand_thr = ix->cand_thr;
  p.thr_init = thr_init;
  p.kprime = kprime;
  p.out_cap = out_cap;
  p.nq = static_cast<int>(nq);
  p.n_rows = N;
  {
    ance::ProfScope ps(ance::kClsCoarse, st);
    ANCE_CUDA((gemm::launch<Ep, BN, STAGES, CG, 4, FMT>(tmA, tmB, ws, p, ctas, st)));
  }
  ance::count_launch(1);
  return ANCE_OK;
}

constexpr int kExactBatch = 1024;  // queries per brute-force pass (bounds the chunk_keys scratch)

int run_exact(ance_index* ix, const float* Q, const int* qlist, int nq, int k, float* D, int64_t* I,
              int64_t row_offset, cudaStream_t st) {
  ExactParams ep;
  ep.Q = Q;
  ep.P = ix->P32;
  ep.d = ix->dim;
  ep.n_rows = ix->n;
  ep.nq_dev = nullptr;
  ep.k = static_cast<int>(std::min<int64_t>(k, std::max<int64_t>(ix->n, 1)));
  ep.k = std::min(ep.k, kMaxK);
  const int sms = gemm::sm_count();
  int n_chunks = static_cast<int>(std::min<int64_t>(2 * sms, (ix->n + 4095) / 4096));
  if (n_chunks < 1) n_chunks = 1;
  ep.n_chunks = n_chunks;
  // the chunk_keys scratch grows with batch * n_chunks * k: above k = 512 the batch shrinks so that it stays the size
  // it has at k = 512 (1.2 GB with 296 chunks)
  const int per_pass = (ep.k <= 512) ? kExactBatch : std::max(1, kExactBatch * 512 / ep.k);
  const int batch = std::min(nq, per_pass);
  int rc = ensure(&ix->chunk_keys, &ix->chunk_keys_elems, static_cast<size_t>(batch) * n_chunks * ep.k);
  if (rc) return rc;
  ep.chunk_keys = ix->chunk_keys;
  const int buf = exact_buf_keys(ep.k);
  const size_t smem = static_cast<size_t>(kExQB) * buf * 8 + static_cast<size_t>(kExQB) * ix->dim * 4;
  void (*chunk)(const ExactParams) = (buf == 1024) ? exact_chunk_kernel<1024>
                                   : (buf == 2048) ? exact_chunk_kernel<2048> : exact_chunk_kernel<4096>;
  static_assert(exact_buf_keys(kMaxK) <= 4096, "exact_chunk_kernel instantiations");
  // per device and cheap: set on every call rather than behind a process-wide flag
  ANCE_CUDA(cudaFuncSetAttribute(chunk, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 static_cast<int>(std::max<size_t>(100 * 1024, smem))));
  for (int b0 = 0; b0 < nq; b0 += per_pass) {
    const int nb = std::min(per_pass, nq - b0);
    ep.qlist = qlist ? qlist + b0 : nullptr;
    ep.q_base = b0;
    ep.nq = nb;
    const int gy = std::max(1, std::min((nb + kExQB - 1) / kExQB, 128));
    ance::ProfScope ps(ance::kClsExact, st);
    chunk<<<dim3(n_chunks, gy), 256, smem, st>>>(ep);
    ANCE_CUDA(cudaGetLastError());
    exact_merge_kernel<<<std::max(1, std::min(nb, 4 * sms)), 256, 0, st>>>(ep, D, I, k, row_offset);
    ANCE_CUDA(cudaGetLastError());
    ance::count_launch(2);
  }
  return ANCE_OK;
}

// One coarse pass + exact rescoring + certificate over `nq` queries whose 16-bit rows are Q16[0..nq);
// qlist (or identity) maps them to rows of q_f32 / D / I.  thr_init == null: tier 1 (running top-k' from -inf, k'
// candidates per split kept).  thr_init != null: tier 2 (start from the per-query threshold, keep everything that
// passes it).  Uncertified queries are appended to flagged_out (+ their next-tier threshold to flagged_thr_out) and
// counted in counters[flag_slot].
int coarse_rescore_pass(ance_index* ix, const uint16_t* Q16, const float* q_f32, int64_t nq, const int* qlist,
                        int kprime, const float* thr_init, int n_splits_req, int k, float* D_dev, int64_t* I_dev,
                        int64_t row_offset, int* flagged_out, float* flagged_thr_out, int flag_slot, int* ns_out,
                        cudaStream_t st) {
  int rc;
  // reservoir size: the smallest that holds about k' more entries between two compactions
  const int cap = reservoir_cap(kprime);
  // tier 2 keeps whatever the reservoir holds at the end (at most cap - 32 entries: a fuller one is compacted at once)
  const int out_cap = thr_init ? cap : kprime;
  // candidates per query, all splits together: the rescore sorts them in shared memory (8 B each)
  const int max_cands = (k <= 512) ? 4096 : kMaxCands;
  const int cg = ix->cta_group;
  const int clusters = (ix->max_ctas > 0 ? ix->max_ctas : gemm::sm_count()) / cg;
  const int q_tiles = static_cast<int>((nq + gemm::BM * cg - 1) / (gemm::BM * cg));
  int n_splits = n_splits_req;
  if (n_splits == 0) {
    // Few query tiles: split the corpus into row ranges so that every CTA (pair) has work, choosing the
    // split count whose work-item count fills whole waves best (ties: fewer splits = fewer candidates).
    n_splits = 1;
    if (q_tiles < 2 * clusters) {
      const int max_splits = std::max(1, std::min(16, max_cands / out_cap));
      double best = -1.0;
      for (int sp = 1; sp <= max_splits; ++sp) {
        const long items = static_cast<long>(q_tiles) * sp;
        const long waves = (items + clusters - 1) / clusters;
        const double eff = static_cast<double>(items) / static_cast<double>(waves * clusters);
        if (eff > best + 1e-9) { best = eff; n_splits = sp; }
      }
    }
  }
  while (n_splits > 1 && n_splits * out_cap > max_cands) --n_splits;
  ANCE_REQUIRE(n_splits * out_cap <= max_cands, "ance_index_search: n_splits * candidates per split = %d exceeds %d",
               n_splits * out_cap, max_cands);
  int ns = 0;
  const bool bf = ix->fmt == ANCE_FMT_BF16;
#define ANCE_COARSE(CG_, CAP_)                                                                                              \
  rc = bf ? launch_coarse<256, (CG_ == 1 ? 4 : 6), CG_, CAP_, tc05::kFmtBF16>(ix, Q16, nq, kprime, out_cap, thr_init, n_splits, &ns, st) \
          : launch_coarse<256, (CG_ == 1 ? 4 : 6), CG_, CAP_, tc05::kFmtF16>(ix, Q16, nq, kprime, out_cap, thr_init, n_splits, &ns, st)
  if (cg == 1 && cap == 1024) { ANCE_COARSE(1, 1024); }
  else if (cg == 1 && cap == 2048) { ANCE_COARSE(1, 2048); }
  else if (cg == 1 && cap == 4096) { ANCE_COARSE(1, 4096); }
  else if (cg == 1) { ANCE_COARSE(1, 8192); }
  else if (cap == 1024) { ANCE_COARSE(2, 1024); }
  else if (cap == 2048) { ANCE_COARSE(2, 2048); }
  else if (cap == 4096) { ANCE_COARSE(2, 4096); }
  else { ANCE_COARSE(2, 8192); }
#undef ANCE_COARSE
  if (rc) return rc;
  *ns_out = ns;
  RescoreParams rp;
  rp.Q = q_f32;
  rp.P = ix->P32;
  rp.d = ix->dim;
  rp.cand_id = ix->cand_id;
  rp.cand_cnt = ix->cand_cnt;
  rp.cand_thr = ix->cand_thr;
  rp.n_splits = ns;
  rp.cand_stride = out_cap;
  rp.k = k;
  rp.qn_hat = ix->qn_hat;
  rp.qn_delta = ix->qn_delta;
  rp.pstats = ix->pstats;
  rp.mu = ix->centred ? ix->mu : nullptr;
  // Accumulation error of the coarse score c = fl(sum_i q^_i p^_i) on the tensor core.  The 16-bit x 16-bit products
  // are exact in fp32; what is unspecified is how tcgen05.mma adds them (PTX: "precision at least that of fp32", order
  // and rounding implementation-defined; published measurements of earlier generations: truncation, block adds of
  // K = 16 aligned to the largest exponent).  Any such scheme performs at most d + d/16 additions, each with an error
  // of at most one ulp of the largest partial sum, 2^-23 * sum_i |q^_i p^_i| <= 2^-23 ||q^|| ||p^|| (Cauchy-Schwarz):
  //   |c - <q^, p^>| <= (17/16) d 2^-23 ||q^|| ||p^||  <  d * 2^-22 * ||q^|| ||p^||          (d = 768: 1.83e-4)
  // tests/test_gpu_search.py measures the real error against an fp64 dot of the same rounded operands (it is ~300x
  // smaller: rounding errors average out, the bound does not assume they do).
  rp.accum_rel = static_cast<float>(ix->dim) * 2.384185791015625e-07f;
  rp.D = D_dev;
  rp.I = I_dev;
  rp.row_offset = row_offset;
  rp.qlist = qlist;
  rp.flagged_list = flagged_out;
  rp.flagged_thr = flagged_thr_out;
  rp.flag_slot = flag_slot;
  rp.counters = ix->counters;
  rp.max_eps = reinterpret_cast<unsigned int*>(ix->counters + 2);
  rp.sort_n = next_pow2(ns * out_cap);
  const size_t rs_smem = static_cast<size_t>(rp.sort_n) * 8 + static_cast<size_t>(ix->dim) * 4 + (ns + 1) * 4 + 16;
  if (rs_smem > 48 * 1024)   // per device and cheap: no process-wide cache
    ANCE_CUDA(cudaFuncSetAttribute(rescore_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(rs_smem)));
  ance::prof_begin(ance::kClsRescore, st);
  rescore_kernel<<<static_cast<unsigned>(nq), 256, rs_smem, st>>>(rp);
  ance::prof_end(ance::kClsRescore, st);
  ANCE_CUDA(cudaGetLastError());
  ance::count_launch(1);
  return ANCE_OK;
}

int create_common(int dim, int64_t capacity_rows, int operand_fmt, float* external_rows, ance_index_t* out) {
  ANCE_REQUIRE(out != nullptr, "ance_index_create: out is null");
  ANCE_REQUIRE(dim > 0 && dim % 8 == 0 && dim <= 4096, "ance_index_create: dim must be a multiple of 8 in (0, 4096], got %d", dim);
  ANCE_REQUIRE(capacity_rows > 0 && capacity_rows < (1ll << 31), "ance_index_create: capacity_rows out of range");
  ANCE_REQUIRE(operand_fmt == ANCE_FMT_BF16 || operand_fmt == ANCE_FMT_FP16, "ance_index_create: bad operand_fmt");
  int rc = check_device();
  if (rc) return rc;
  ance_index* ix = new ance_index();
  ix->dim = dim;
  ix->cap = capacity_rows;
  ix->fmt = operand_fmt;
  cudaGetDevice(&ix->device);
  const size_t elems = static_cast<size_t>(capacity_rows) * dim;
  cudaError_t e1 = cudaSuccess;
  if (external_rows) {
    ix->P32 = external_rows;
    ix->owns_p32 = false;
  } else {
    e1 = cudaMalloc(&ix->P32, elems * 4);
  }
  cudaError_t e2 = cudaMalloc(&ix->P16, elems * 2);
  cudaError_t e3 = cudaMalloc(&ix->pstats, 2 * sizeof(unsigned int));
  cudaError_t e4 = cudaMalloc(&ix->pace, kMaxPace * sizeof(int));
  cudaError_t e5 = cudaMalloc(&ix->counters, kNumCounters * sizeof(int));
  cudaError_t e6 = cudaMalloc(&ix->mu, static_cast<size_t>(dim) * sizeof(float));
  cudaError_t e7 = cudaMalloc(&ix->colsum, static_cast<size_t>(dim) * sizeof(double));
  if (e1 || e2 || e3 || e4 || e5 || e6 || e7) {
    ance::set_error("ance_index_create: cudaMalloc failed for %lld x %d rows", (long long)capacity_rows, dim);
    ance_index_destroy(ix);
    return ANCE_ERR_NOMEM;
  }
  cudaMemset(ix->pstats, 0, 2 * sizeof(unsigned int));
  cudaMemset(ix->counters, 0, kNumCounters * sizeof(int));
  *out = ix;
  return ANCE_OK;
}

// (Re)build the 16-bit operands of every row from the fp32 rows: column mean -> centre -> round, norm maxima, range flag.
// Runs once per index state (lazily, at the first search after rows were added): ~45 GB of HBM traffic for 8.84M rows,
// about 10 ms — nothing next to the encode that produced the rows — and it lets the centre be the mean of ALL rows.
int prepare_operands(ance_index* ix, cudaStream_t st) {
  if (!ix->dirty) return ANCE_OK;
  const int64_t n = ix->n;
  ANCE_CUDA(cudaMemsetAsync(ix->pstats, 0, 2 * sizeof(unsigned int), st));
  ANCE_CUDA(cudaMemsetAsync(ix->counters + kCntRowErr, 0, sizeof(int), st));
  ance::ProfScope ps(ance::kClsQuant, st);
  ix->centred = ix->center && n >= 256;
  if (ix->centred) {
    ANCE_CUDA(cudaMemsetAsync(ix->colsum, 0, static_cast<size_t>(ix->dim) * sizeof(double), st));
    // rows per block: enough blocks to fill the machine for a small index, few enough atomics (n / slab per column) for a big one
    const int slab = static_cast<int>(std::min<int64_t>(4096, std::max<int64_t>(32, n / (8 * gemm::sm_count()))));
    column_sum_kernel<<<static_cast<unsigned>((n + slab - 1) / slab), 256, 0, st>>>(ix->P32, n, ix->dim, slab, ix->colsum);
    finalize_mean_kernel<<<(ix->dim + 255) / 256, 256, 0, st>>>(ix->colsum, n, ix->dim, ix->mu);
    ANCE_CUDA(cudaGetLastError());
    ance::count_launch(2);
  }
  const float* mu = ix->centred ? ix->mu : nullptr;
  const int wpb = 8;
  const unsigned blocks = static_cast<unsigned>((n + wpb - 1) / wpb);
  if (n > 0) {
    if (ix->fmt == ANCE_FMT_BF16)
      quantize_rows_kernel<true><<<blocks, wpb * 32, 0, st>>>(ix->P32, ix->P16, n, ix->dim, mu, nullptr, nullptr, ix->pstats, ix->counters + kCntRowErr);
    else
      quantize_rows_kernel<false><<<blocks, wpb * 32, 0, st>>>(ix->P32, ix->P16, n, ix->dim, mu, nullptr, nullptr, ix->pstats, ix->counters + kCntRowErr);
    ANCE_CUDA(cudaGetLastError());
    ance::count_launch(1);
  }
  ix->dirty = false;
  return ANCE_OK;
}

}  // namespace

extern "C" int ance_index_create(int dim, int64_t capacity_rows, int operand_fmt, ance_index_t* out) {
  return create_common(dim, capacity_rows, operand_fmt, nullptr, out);
}

extern "C" int ance_index_create_over(int dim, int64_t capacity_rows, int operand_fmt, float* rows_dev,
                                      ance_index_t* out) {
  ANCE_REQUIRE(rows_dev != nullptr, "ance_index_create_over: rows_dev is null");
  ANCE_REQUIRE((reinterpret_cast<uintptr_t>(rows_dev) & 15) == 0, "ance_index_create_over: rows_dev must be 16-byte aligned");
  return create_common(dim, capacity_rows, operand_fmt, rows_dev, out);
}

extern "C" int ance_index_destroy(ance_index_t ix) {
  if (!ix) return ANCE_OK;
  void* ptrs[] = {ix->owns_p32 ? ix->P32 : nullptr, ix->P16, ix->pstats, ix->Q16, ix->qn_hat, ix->qn_delta, ix->scratch_sc,
                  ix->scratch_id, ix->cand_id, ix->cand_cnt, ix->cand_thr, ix->flagged, ix->flagged_thr, ix->counters,
                  ix->chunk_keys, ix->flagged2, ix->Q16b, ix->pace, ix->mu, ix->colsum};
  for (void* p : ptrs)
    if (p) cudaFree(p);
  delete ix;
  return ANCE_OK;
}

extern "C" int ance_index_reset(ance_index_t ix) {
  ANCE_REQUIRE(ix != nullptr, "ance_index_reset: null handle");
  ix->n = 0;
  ix->dirty = false;
  ANCE_CUDA(cudaMemset(ix->pstats, 0, 2 * sizeof(unsigned int)));
  ANCE_CUDA(cudaMemset(ix->counters, 0, kNumCounters * sizeof(int)));
  return ANCE_OK;
}

extern "C" int64_t ance_index_ntotal(ance_index_t ix) { return ix ? ix->n : -1; }

extern "C" int ance_index_add(ance_index_t ix, const float* rows_dev, int64_t n, void* stream) {
  ANCE_REQUIRE(ix != nullptr, "ance_index_add: null handle");
  ANCE_REQUIRE(n >= 0, "ance_index_add: negative row count");
  if (n == 0) return ANCE_OK;
  ANCE_REQUIRE(rows_dev != nullptr, "ance_index_add: rows_dev is null");
  ANCE_REQUIRE(ix->n + n <= ix->cap, "ance_index_add: %lld + %lld rows exceed capacity %lld", (long long)ix->n,
               (long long)n, (long long)ix->cap);
  int rc = check_handle_device(ix, "ance_index_add");
  if (rc) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  float* dst = ix->P32 + static_cast<size_t>(ix->n) * ix->dim;
  if (dst != rows_dev)   // rows produced in place (the encoder wrote straight into the index storage): no copy
    ANCE_CUDA(cudaMemcpyAsync(dst, rows_dev, static_cast<size_t>(n) * ix->dim * 4, cudaMemcpyDeviceToDevice, st));
  ix->n += n;
  ix->dirty = true;      // the 16-bit operands are (re)built from all rows by the next ance_index_prepare / search
  return ANCE_OK;
}

extern "C" int ance_index_prepare(ance_index_t ix, void* stream) {
  ANCE_REQUIRE(ix != nullptr, "ance_index_prepare: null handle");
  int rc = check_handle_device(ix, "ance_index_prepare");
  if (rc) return rc;
  return prepare_operands(ix, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int ance_index_set_param(ance_index_t ix, const char* name, double value) {
  ANCE_REQUIRE(ix != nullptr && name != nullptr, "ance_index_set_param: null argument");
  const int v = static_cast<int>(value);
  if (!strcmp(name, "kprime")) {
    ANCE_REQUIRE(v >= 0 && v <= kMaxKprime && v % 32 == 0, "kprime must be a multiple of 32 in [0, %d]", kMaxKprime);
    ix->kprime = v;
  }
  else if (!strcmp(name, "n_splits")) { ANCE_REQUIRE(v >= 0 && v <= 64, "n_splits must be in [0, 64]"); ix->n_splits = v; }
  else if (!strcmp(name, "cta_group")) { ANCE_REQUIRE(v == 1 || v == 2, "cta_group must be 1 or 2"); ix->cta_group = v; }
  else if (!strcmp(name, "exact_fallback")) { ix->exact_fallback = v != 0; }
  else if (!strcmp(name, "tier2")) { ix->tier2 = v != 0; }
  else if (!strcmp(name, "max_ctas")) { ANCE_REQUIRE(v >= 0, "max_ctas must be >= 0"); ix->max_ctas = v; }
  else if (!strcmp(name, "pace_window")) { ANCE_REQUIRE(v >= 0 && v <= 4096, "pace_window must be in [0, 4096]"); ix->pace_window = v; }
  else if (!strcmp(name, "operand_fmt")) {
    // re-round the rows already in the index to the other 16-bit format (the fp32 rows are kept for exactly this)
    ANCE_REQUIRE(v == ANCE_FMT_BF16 || v == ANCE_FMT_FP16, "operand_fmt must be ANCE_FMT_FP16 or ANCE_FMT_BF16");
    int rc = check_handle_device(ix, "ance_index_set_param");
    if (rc) return rc;
    if (v != ix->fmt) {
      ix->fmt = v;
      ix->dirty = true;
    }
  }
  else if (!strcmp(name, "center")) { ix->center = v != 0; ix->dirty = true; }
  else { ance::set_error("ance_index_set_param: unknown parameter '%s'", name); return ANCE_ERR_INVALID; }
  return ANCE_OK;
}

extern "C" int ance_index_search_exact(ance_index_t ix, const float* q_dev, int64_t nq, int k, float* D_dev,
                                       int64_t* I_dev, int64_t row_offset, void* stream) {
  ANCE_REQUIRE(ix != nullptr, "ance_index_search_exact: null handle");
  ANCE_REQUIRE(nq >= 0 && k > 0, "ance_index_search_exact: need nq >= 0 and k > 0");
  ANCE_REQUIRE(k <= kMaxK, "ance_index_search_exact: k = %d exceeds the largest supported k, %d", k, kMaxK);
  if (nq == 0) return ANCE_OK;
  ANCE_REQUIRE(q_dev && D_dev && I_dev, "ance_index_search_exact: null buffer");
  int rc = check_handle_device(ix, "ance_index_search_exact");
  if (rc) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (ix->n == 0) {
    // faiss on an empty index: labels -1, scores lowest float
    std::vector<float> d(static_cast<size_t>(nq) * k, -FLT_MAX);
    std::vector<int64_t> i(static_cast<size_t>(nq) * k, -1);
    ANCE_CUDA(cudaMemcpyAsync(D_dev, d.data(), d.size() * 4, cudaMemcpyHostToDevice, st));
    ANCE_CUDA(cudaMemcpyAsync(I_dev, i.data(), i.size() * 8, cudaMemcpyHostToDevice, st));
    ANCE_CUDA(cudaStreamSynchronize(st));
    return ANCE_OK;
  }
  return run_exact(ix, q_dev, nullptr, static_cast<int>(nq), k, D_dev, I_dev, row_offset, st);
}

extern "C" int ance_index_search(ance_index_t ix, const float* q_dev, int64_t nq, int k, float* D_dev,
                                 int64_t* I_dev, int64_t row_offset, void* stream) {
  ANCE_REQUIRE(ix != nullptr, "ance_index_search: null handle");
  ANCE_REQUIRE(nq >= 0 && nq < (1ll << 31), "ance_index_search: nq out of range");
  ANCE_REQUIRE(k > 0, "ance_index_search: k must be positive");
  ANCE_REQUIRE(k <= kMaxK, "ance_index_search: k = %d exceeds the largest supported k, %d", k, kMaxK);
  if (nq == 0) return ANCE_OK;
  ANCE_REQUIRE(q_dev && D_dev && I_dev, "ance_index_search: null buffer");
  int rc = check_handle_device(ix, "ance_index_search");
  if (rc) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  // choose k' (candidates kept per split).  The certificate needs every row within eps of the k-th score among the
  // candidates; eps is ~0.5 (fp16 operands) / ~3 (bf16) for rows of norm 27.7, i.e. ~0.1 k / ~0.6 k extra rows on the
  // distributions of tools/exp_certify.py.  A query that k' does not cover costs one tier-2 pass, not a wrong answer.
  // k > 512 (up to kMaxK): the same formulas without the caps, served by the large reservoirs (reservoir_cap).
  int kprime = ix->kprime;
  if (kprime == 0) {
    const int want = (ix->fmt == ANCE_FMT_FP16) ? k + k / 2 - k / 16 : 2 * k + 32;   // fp16: ~1.44 k (k = 200: 288)
    if (k <= 240) kprime = std::min(512, std::max(64, (want + 31) / 32 * 32));
    else if (k <= 512) kprime = std::min(992, (2 * k + 31) / 32 * 32);
    else kprime = (want + 31) / 32 * 32;   // k = 1000: 1440 (fp16) / 2048 (bf16); k = 2048: 2944 / 4128
  }
  const bool small_k = k <= 512;
  if (kprime < k || (small_k && kprime > 992) || ix->n < 4 * static_cast<int64_t>(kprime)) {
    // tiny index (or a k' set below k): the exact brute-force path is both correct and cheap enough
    ix->stats = ance_search_stats{};
    ix->stats.nq = nq;
    ix->stats.n_uncertified = nq;
    return ance_index_search_exact(ix, q_dev, nq, k, D_dev, I_dev, row_offset, stream);
  }
  if ((rc = prepare_operands(ix, st))) return rc;
  // --- 1. quantize queries
  {
    size_t a = static_cast<size_t>(ix->q_cap) * ix->dim, b = ix->q_cap, c = ix->q_cap;
    if ((rc = ensure(&ix->Q16, &a, static_cast<size_t>(nq) * ix->dim))) return rc;
    if ((rc = ensure(&ix->qn_hat, &b, static_cast<size_t>(nq)))) return rc;
    if ((rc = ensure(&ix->qn_delta, &c, static_cast<size_t>(nq)))) return rc;
    ix->q_cap = std::max<int64_t>(ix->q_cap, nq);
    size_t f = ix->flagged_cap, g = ix->flagged_cap;
    if ((rc = ensure(&ix->flagged, &f, static_cast<size_t>(nq)))) return rc;
    if ((rc = ensure(&ix->flagged_thr, &g, static_cast<size_t>(nq)))) return rc;
    ix->flagged_cap = f;
  }
  ANCE_CUDA(cudaMemsetAsync(ix->counters, 0, kCntRowErr * sizeof(int), st));   // everything but the sticky row flag
  const unsigned qblocks = static_cast<unsigned>((nq + 7) / 8);
  ance::prof_begin(ance::kClsQuant, st);
  if (ix->fmt == ANCE_FMT_BF16)
    quantize_rows_kernel<true><<<qblocks, 256, 0, st>>>(q_dev, ix->Q16, nq, ix->dim, nullptr, ix->qn_hat, ix->qn_delta, nullptr, ix->counters + kCntQueryErr);
  else
    quantize_rows_kernel<false><<<qblocks, 256, 0, st>>>(q_dev, ix->Q16, nq, ix->dim, nullptr, ix->qn_hat, ix->qn_delta, nullptr, ix->counters + kCntQueryErr);
  ance::prof_end(ance::kClsQuant, st);
  ANCE_CUDA(cudaGetLastError());
  ance::count_launch(1);
  // --- 2+3. tier 1: coarse pass over all queries, exact rescoring, certificate
  int ns = 0;
  rc = coarse_rescore_pass(ix, ix->Q16, q_dev, nq, nullptr, kprime, nullptr, ix->n_splits, k, D_dev, I_dev, row_offset,
                           ix->flagged, ix->flagged_thr, 0, &ns, st);
  if (rc) return rc;
  // One small D2H + sync per search tells the host how many queries stay uncertified and whether an operand left
  // the 16-bit format's range (the reference's search call is synchronous as well).
  int h[kNumCounters] = {};
  ANCE_CUDA(cudaMemcpyAsync(h, ix->counters, sizeof(h), cudaMemcpyDeviceToHost, st));
  ANCE_CUDA(cudaStreamSynchronize(st));
  if (h[kCntQueryErr] || h[kCntRowErr]) {
    // coarse scores, thresholds and the certificate would be compared against inf / NaN: refuse instead of
    // returning ANCE_OK with unverifiable neighbours
    ance::set_error("ance_index_search: %s non-finite after rounding to %s (inf / NaN in the input%s)",
                    h[kCntRowErr] ? "an index row is" : "a query is", ix->fmt == ANCE_FMT_FP16 ? "fp16" : "bf16",
                    ix->fmt == ANCE_FMT_FP16 ? ", or |x| > 65504: switch with ance_index_set_param(\"operand_fmt\", ANCE_FMT_BF16)" : "");
    return ANCE_ERR_UNSUPPORTED;
  }
  int n_exact = h[0];
  int ns2 = 0;
  const int kprime2 = tier2_kprime(k);
  if (h[0] > 0 && ix->tier2 && ix->n >= 4 * static_cast<int64_t>(kprime2)) {
    // --- tier 2: the uncertified queries once more, from their own thresholds (nothing that passes is dropped)
    const int n2 = h[0];
    if ((rc = ensure(&ix->Q16b, &ix->q16b_elems, static_cast<size_t>(n2) * ix->dim))) return rc;
    if ((rc = ensure(&ix->flagged2, &ix->flagged2_cap, static_cast<size_t>(n2)))) return rc;
    gather_rows16_kernel<<<n2, 96, 0, st>>>(ix->Q16, ix->flagged, n2, ix->dim, ix->Q16b);
    ANCE_CUDA(cudaGetLastError());
    ance::count_launch(1);
    rc = coarse_rescore_pass(ix, ix->Q16b, q_dev, n2, ix->flagged, kprime2, ix->flagged_thr, 0, k, D_dev, I_dev, row_offset,
                             ix->flagged2, nullptr, 3, &ns2, st);
    if (rc) return rc;
    ANCE_CUDA(cudaMemcpyAsync(h, ix->counters, sizeof(h), cudaMemcpyDeviceToHost, st));
    ANCE_CUDA(cudaStreamSynchronize(st));
    n_exact = h[3];
    if (n_exact > 0 && ix->exact_fallback) {
      rc = run_exact(ix, q_dev, ix->flagged2, n_exact, k, D_dev, I_dev, row_offset, st);
      if (rc) return rc;
    }
  } else if (n_exact > 0 && ix->exact_fallback) {
    // --- tier 3: exact brute force
    rc = run_exact(ix, q_dev, ix->flagged, n_exact, k, D_dev, I_dev, row_offset, st);
    if (rc) return rc;
  }
  ix->stats = ance_search_stats{};
  ix->stats.nq = nq;
  ix->stats.kprime = kprime;
  ix->stats.n_splits = ns;
  ix->stats.n_tier2 = h[0];
  ix->stats.n_uncertified = n_exact;
  ix->stats.n_candidates = h[1];
  memcpy(&ix->stats.max_eps, &h[2], 4);
  ix->last_stream = st;
  return ANCE_OK;
}

extern "C" int ance_index_last_stats(ance_index_t ix, ance_search_stats* out) {
  ANCE_REQUIRE(ix != nullptr && out != nullptr, "ance_index_last_stats: null argument");
  *out = ix->stats;
  return ANCE_OK;
}
