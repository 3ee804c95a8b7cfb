// Top-k serving epilogue over full-catalogue scores (SURVEY.md section 8f-4): for every batch row
// the k best catalogue columns, so that k (column, score) pairs leave the device instead of the
// whole [rows, N] matrix. One CTA per row, exact and deterministic (score descending, ties by
// ascending column):
//   1. pivot from a sample: 1024 strided scores are sorted in shared memory; the pivot is the
//      sample of the rank that leaves ~3k + slack scores above it;
//   2. ONE sweep over the row appends every score >= pivot to a candidate list in shared memory
//      (<= 4096 entries: a few hundred in practice);
//   3. exact radix select (11 + 11 + 10 bits of the order-preserving key) over the candidates
//      finds the k-th largest key T and how many entries equal to T still belong to the top k;
//   4. the winners are collected and ordered by a bitonic sort of <= 512 slots.
// When the sample misleads (fewer than k or more than 4096 candidates) the radix select runs over
// the whole row instead (three more sweeps), and when entries tie with T beyond what fits, the
// ties are taken in column order by an ordered sweep of the row - both rare, both exact.
#pragma once

#include "ocf_kernels.cuh"

namespace ocf {

constexpr int TOPK_MAX = 512;
constexpr int TOPK_THREADS = 256;
constexpr int TOPK_SAMPLE = 1024;
constexpr int TOPK_CAND = 4096;

__device__ __forceinline__ uint32_t score_key(float x) {
  const uint32_t u = __float_as_uint(x);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key_score(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// Seen items never come back as recommendations: the row's input entries get score -inf.
__global__ void __launch_bounds__(128) k_exclude_inputs(BatchDev bt, float* __restrict__ scores, long long ldo) {
  const int4 it = bt.items[blockIdx.x];
  const int p0 = bt.ent_off[it.x] + it.y;
  for (int i = threadIdx.x; i < it.z; i += 128)
    if (bt.codes[p0 + i] & CODE_IN) scores[(long long)it.x * ldo + bt.ent_col[p0 + i]] = -INFINITY;
}

// Largest bin b with  (entries in bins > b) < need <= (entries in bins >= b); one warp, `nb` bins
// (a multiple of 32). Leaves b, the count above it and the count in it.
__device__ __forceinline__ void find_bin(const int* __restrict__ hist, int nb, int need, int* bin, int* above, int* inside) {
  const int lane = threadIdx.x & 31, per = nb / 32;
  int own = 0;                                     // lane l owns bins [l*per, (l+1)*per)
  for (int i = 0; i < per; ++i) own += hist[lane * per + i];
  int suf = own;                                   // inclusive suffix sum over the lanes
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_down_sync(FULL, suf, o); if (lane + o < 32) suf += t; }
  const int higher = suf - own;
  if (higher < need && need <= suf) {              // the crossing is inside this lane's bins
    int acc = higher;
    for (int i = per - 1; i >= 0; --i) {
      const int h = hist[lane * per + i];
      if (acc + h >= need) { *bin = lane * per + i; *above = acc; *inside = h; break; }
      acc += h;
    }
  }
}

// Bitonic sort of n (a power of two) (key, col) slots in shared memory: key descending, column ascending.
// `payload` (optional) moves with its slot.
__device__ __forceinline__ void bitonic_desc(uint32_t* key, int32_t* col, int n, bool with_col, int32_t* payload = nullptr) {
  for (int size = 2; size <= n; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = threadIdx.x; t < n / 2; t += TOPK_THREADS) {
        const int lo = 2 * t - (t & (stride - 1)), hi = lo + stride;
        const bool up = (lo & size) == 0;
        const uint32_t ka = key[lo], kb = key[hi];
        const int32_t ca = with_col ? col[lo] : 0, cb = with_col ? col[hi] : 0;
        const bool a_first = ka > kb || (ka == kb && ca < cb);
        if (a_first != up) {
          key[lo] = kb; key[hi] = ka;
          if (with_col) { col[lo] = cb; col[hi] = ca; }
          if (payload) { const int32_t p = payload[lo]; payload[lo] = payload[hi]; payload[hi] = p; }
        }
      }
      __syncthreads();
    }
  }
}

__global__ void __launch_bounds__(TOPK_THREADS)
k_topk(const float* __restrict__ scores, long long ldo, int n_cols, int k,
       int32_t* __restrict__ out_cols, float* __restrict__ out_scores) {
  __shared__ int hist[2048];
  __shared__ uint32_t c_key[TOPK_CAND];            // sample first, then the candidates
  __shared__ int32_t c_col[TOPK_CAND];
  __shared__ uint32_t w_key[TOPK_MAX];
  __shared__ int32_t w_col[TOPK_MAX];
  __shared__ int s_bin, s_above, s_inside, s_count, s_taken, s_ties;
  __shared__ int s_wcnt[TOPK_THREADS / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float* row = scores + (long long)blockIdx.x * ldo;
  const int kk = min(min(k, n_cols), TOPK_MAX);

  // ---- 1. pivot ----------------------------------------------------------------------------------
  uint32_t pivot = 0u;                             // key 0 = below every score: small rows take everything
  if (n_cols > TOPK_CAND) {
    for (int j = tid; j < TOPK_SAMPLE; j += TOPK_THREADS)
      c_key[j] = score_key(__ldcg(row + (long long)j * n_cols / TOPK_SAMPLE));
    __syncthreads();
    bitonic_desc(c_key, c_col, TOPK_SAMPLE, false);
    const long long r = 3LL * kk * TOPK_SAMPLE / n_cols + 8;          // ~3k + slack of the row above the pivot
    pivot = c_key[r < TOPK_SAMPLE ? (int)r : TOPK_SAMPLE - 1];
    __syncthreads();
  }
  // ---- 2. candidates: every score >= pivot --------------------------------------------------------
  if (tid == 0) s_count = 0;
  __syncthreads();
  for (int i = tid; i < n_cols; i += TOPK_THREADS) {
    const uint32_t key = score_key(__ldcg(row + i));
    if (key >= pivot) {
      const int slot = atomicAdd(&s_count, 1);
      if (slot < TOPK_CAND) { c_key[slot] = key; c_col[slot] = i; }
    }
  }
  __syncthreads();
  const int n_cand = s_count;
  const bool from_row = n_cand < kk || n_cand > TOPK_CAND;            // the sample misled: select over the whole row
  const int n_src = from_row ? n_cols : n_cand;
  // ---- 3. exact radix select of the k-th largest key over the source -------------------------------
  uint32_t prefix = 0;
  int need = kk, ties_total = 0;
  for (int level = 0; level < 3; ++level) {
    const int shift = level == 0 ? 21 : (level == 1 ? 10 : 0);
    const int nb = level == 2 ? 1024 : 2048;
    for (int i = tid; i < 2048; i += TOPK_THREADS) hist[i] = 0;
    __syncthreads();
    for (int i = tid; i < n_src; i += TOPK_THREADS) {
      const uint32_t key = from_row ? score_key(__ldcg(row + i)) : c_key[i];
      const bool in = level == 0 || (level == 1 ? (key >> 21) == (prefix >> 21) : (key >> 10) == (prefix >> 10));
      if (in) {
        const int bin = (int)((key >> shift) & (uint32_t)(nb - 1));
        const unsigned same = __match_any_sync(__activemask(), bin);   // scores cluster: one atomic per distinct bin and warp
        if (lane == __ffs(same) - 1) atomicAdd(&hist[bin], __popc(same));
      }
    }
    __syncthreads();
    if (warp == 0) find_bin(hist, nb, need, &s_bin, &s_above, &s_inside);
    __syncthreads();
    prefix |= (uint32_t)s_bin << shift;
    need -= s_above;
    ties_total = s_inside;
    __syncthreads();
  }
  const uint32_t T = prefix;                       // the k-th largest key; `need` of the `ties_total` entries equal to T are taken
  // ---- 4. winners ------------------------------------------------------------------------------------
  if (tid == 0) { s_taken = 0; s_ties = 0; }
  __syncthreads();
  if (!from_row && ties_total == need) {
    // every tie is a winner: no order needed among the candidates
    for (int i = tid; i < n_cand; i += TOPK_THREADS) {
      const uint32_t key = c_key[i];
      if (key >= T) { const int slot = atomicAdd(&s_taken, 1); w_key[slot] = key; w_col[slot] = c_col[i]; }
    }
  } else {
    // ordered sweep of the row: key > T in any order, the first `need` ties in column order
    for (int i0 = 0; i0 < n_cols; i0 += TOPK_THREADS) {
      const int i = i0 + tid;
      const uint32_t key = i < n_cols ? score_key(__ldcg(row + i)) : 0u;
      const bool tie = i < n_cols && key == T;
      if (i < n_cols && key > T) { const int slot = atomicAdd(&s_taken, 1); w_key[slot] = key; w_col[slot] = i; }
      const unsigned tm = __ballot_sync(FULL, tie);
      if (lane == 0) s_wcnt[warp] = __popc(tm);
      const int any = __syncthreads_or(tie ? 1 : 0);
      if (any) {
        int before = s_ties;
        for (int w = 0; w < warp; ++w) before += s_wcnt[w];
        const int rank = before + __popc(tm & ((1u << lane) - 1u));
        if (tie && rank < need) { const int slot = atomicAdd(&s_taken, 1); w_key[slot] = key; w_col[slot] = i; }
        __syncthreads();
        if (tid == 0) { int t = 0; for (int w = 0; w < TOPK_THREADS / 32; ++w) t += s_wcnt[w]; s_ties += t; }
        __syncthreads();
      }
    }
  }
  __syncthreads();
  for (int i = s_taken + tid; i < TOPK_MAX; i += TOPK_THREADS) { w_key[i] = 0u; w_col[i] = 0x7fffffff; }
  __syncthreads();
  bitonic_desc(w_key, w_col, TOPK_MAX, true);
  for (int j = tid; j < k; j += TOPK_THREADS) {
    const bool ok = j < kk && w_key[j] != 0u;
    const float sc = ok ? key_score(w_key[j]) : -INFINITY;
    out_cols[(long long)blockIdx.x * k + j] = (ok && sc != -INFINITY) ? w_col[j] : -1;
    out_scores[(long long)blockIdx.x * k + j] = sc;
  }
}

}  // namespace ocf
