// Ranking evaluation over full-catalogue scores (DESIGN.md section 2, row f-5): for every relevant
// target of a batch row, its exact 1-based rank among the row's candidate columns in the order of
// k_topk (score descending, ties by ascending column). One read of the [rows, N] score matrix that
// ocf_score left in HBM:
//   1. k_rank_prep (one CTA per row): the row's relevant targets (CODE_TGT, stored value >= min_value,
//      score not -inf after k_exclude_inputs), compacted in entry order into the workspace at the row's
//      entry offset, then every chunk of RANK_CHUNK of them sorted best first in shared memory;
//   2. k_rank_count (grid slices x rows): each CTA holds one chunk's sorted keys in shared memory and
//      sweeps its slice of the score row once. A candidate below the chunk's worst target (the common
//      case) only bumps a register; any other finds by binary search how many chunk targets are ahead
//      of it (pos) and adds 1 to hist[pos]. The histogram goes to per-target counters with integer
//      atomics. Rows with more than one chunk sweep the slice once per chunk;
//   3. k_rank_finish (one CTA per row): target j of a chunk has rank = hist[0] + ... + hist[j] summed
//      over the slices (the candidates ahead of it, plus itself). Ranks are scattered back to entry
//      order; every other entry gets 0.
// Every count is an integer, so the ranks do not depend on the grid shape or the order of the atomics.
#pragma once

#include "ocf_topk.cuh"

namespace ocf {

constexpr int RANK_THREADS = TOPK_THREADS;       // bitonic_desc strides by TOPK_THREADS
constexpr int RANK_CHUNK = 2048;                 // relevant targets per shared-memory chunk

struct RankArgs {
  BatchDev bt;
  const float* scores;       // [rows, ldo] after k_exclude_inputs
  long long ldo;
  int n_cols;
  float min_value;
  int slice_len;             // columns per k_rank_count CTA (a multiple of 4)
  uint32_t* key;             // [max_entries] a row's relevant targets from ent_off[b] on, each chunk sorted best first
  int32_t* col;
  int32_t* ent;              //   their entry index
  int32_t* cnt;              //   candidates with exactly j chunk targets ahead of them, for target j of its chunk
  int32_t* n_rel;            // [rows]
  unsigned long long* n_cand;// [rows] columns with a finite score
  int32_t* rank;             // [max_entries] per entry: 1-based rank, 0 = not a relevant target
};

// Inclusive block-wide prefix sum of one int per thread (RANK_THREADS threads); `tot` gets the block total.
__device__ __forceinline__ int block_scan_incl(int v, int* s_warp, int* tot) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(FULL, v, o); if (lane >= o) v += t; }
  if (lane == 31) s_warp[warp] = v;
  __syncthreads();
  int before = 0, all = 0;
#pragma unroll
  for (int w = 0; w < RANK_THREADS / 32; ++w) { const int x = s_warp[w]; before += w < warp ? x : 0; all += x; }
  __syncthreads();
  *tot = all;
  return v + before;
}

__global__ void __launch_bounds__(RANK_THREADS) k_rank_prep(RankArgs a) {
  __shared__ uint32_t s_key[RANK_CHUNK];
  __shared__ int32_t s_col[RANK_CHUNK];
  __shared__ int32_t s_ent[RANK_CHUNK];
  __shared__ int s_warp[RANK_THREADS / 32];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int p0 = a.bt.ent_off[b], p1 = a.bt.ent_off[b + 1];
  const float* row = a.scores + (long long)b * a.ldo;
  // ---- relevant targets, compacted in entry order --------------------------------------------------
  int n = 0;
  for (int i0 = p0; i0 < p1; i0 += RANK_THREADS) {
    const int i = i0 + tid;
    int rel = 0; uint32_t k = 0u; int32_t c = 0;
    if (i < p1 && (a.bt.codes[i] & CODE_TGT) && a.bt.ent_val[i] >= a.min_value) {
      c = a.bt.ent_col[i];
      const float s = row[c];
      if (s != -INFINITY) { rel = 1; k = score_key(s); }
    }
    int tot;
    const int at = block_scan_incl(rel, s_warp, &tot) - rel;
    if (rel) { a.key[p0 + n + at] = k; a.col[p0 + n + at] = c; a.ent[p0 + n + at] = i; a.cnt[p0 + n + at] = 0; }
    n += tot;
  }
  if (tid == 0) { a.n_rel[b] = n; a.n_cand[b] = 0ull; }
  // ---- every chunk sorted best first (score key descending, column ascending) -----------------------
  for (int c0 = 0; c0 < n; c0 += RANK_CHUNK) {
    const int len = min(RANK_CHUNK, n - c0);
    if (len > 1) {
      int m = 2;
      while (m < len) m <<= 1;
      __syncthreads();                             // this thread's compaction writes / the previous chunk's reads are done
      for (int j = tid; j < m; j += RANK_THREADS) {
        const bool in = j < len;
        s_key[j] = in ? a.key[p0 + c0 + j] : 0u;   // key 0 sorts after every finite score
        s_col[j] = in ? a.col[p0 + c0 + j] : 0x7fffffff;
        s_ent[j] = in ? a.ent[p0 + c0 + j] : -1;
      }
      __syncthreads();
      bitonic_desc(s_key, s_col, m, true, s_ent);
      for (int j = tid; j < len; j += RANK_THREADS) {
        a.key[p0 + c0 + j] = s_key[j]; a.col[p0 + c0 + j] = s_col[j]; a.ent[p0 + c0 + j] = s_ent[j];
      }
    }
  }
}

__global__ void __launch_bounds__(RANK_THREADS) k_rank_count(RankArgs a) {
  __shared__ uint32_t s_key[RANK_CHUNK];
  __shared__ int32_t s_col[RANK_CHUNK];
  __shared__ int hist[RANK_CHUNK];
  __shared__ int s_warp[RANK_THREADS / 32];
  const int b = blockIdx.y, tid = threadIdx.x;
  const int lo = blockIdx.x * a.slice_len, hi = min(lo + a.slice_len, a.n_cols);
  if (lo >= hi) return;
  const int n = a.n_rel[b];
  const int base = a.bt.ent_off[b];
  const long long off = (long long)b * a.ldo;
  const float* row = a.scores + off;
  const int head = min((int)((4 - (off + lo) % 4) % 4), hi - lo);   // scalar columns up to a 16-byte boundary
  const int v0 = lo + head, nvec = (hi - v0) >> 2;
  const float4* vrow = reinterpret_cast<const float4*>(row + v0);
  const int nch = max(1, (n + RANK_CHUNK - 1) / RANK_CHUNK);    // a row without targets still counts its candidates
  for (int ch = 0; ch < nch; ++ch) {
    const int c0 = ch * RANK_CHUNK, len = min(RANK_CHUNK, n - c0);
    for (int j = tid; j < len; j += RANK_THREADS) { s_key[j] = a.key[base + c0 + j]; s_col[j] = a.col[base + c0 + j]; hist[j] = 0; }
    __syncthreads();
    // a candidate (key, column) is below every target of the chunk when it is behind the last one
    const uint32_t wk = len > 0 ? s_key[len - 1] : 0xffffffffu;
    const int wc = len > 0 ? s_col[len - 1] : -1;
    int cand = 0;
    auto visit = [&](int j, float s) {
      if (s == -INFINITY) return;
      ++cand;
      const uint32_t k = score_key(s);
      if (k < wk || (k == wk && j > wc)) return;
      int l = 0, r = len - 1;                      // targets [0, l) are ahead; the last one is not
      while (l < r) {
        const int mid = (l + r) >> 1;
        const uint32_t mk = s_key[mid];
        if (mk > k || (mk == k && s_col[mid] < j)) l = mid + 1; else r = mid;
      }
      atomicAdd(&hist[l], 1);
    };
    if (tid < head) visit(lo + tid, __ldcg(row + lo + tid));
    int q = tid;
    for (; q + RANK_THREADS < nvec; q += 2 * RANK_THREADS) {
      const float4 x = __ldcg(vrow + q), y = __ldcg(vrow + q + RANK_THREADS);
      const int j = v0 + 4 * q, jy = j + 4 * RANK_THREADS;
      visit(j, x.x); visit(j + 1, x.y); visit(j + 2, x.z); visit(j + 3, x.w);
      visit(jy, y.x); visit(jy + 1, y.y); visit(jy + 2, y.z); visit(jy + 3, y.w);
    }
    if (q < nvec) {
      const float4 x = __ldcg(vrow + q);
      const int j = v0 + 4 * q;
      visit(j, x.x); visit(j + 1, x.y); visit(j + 2, x.z); visit(j + 3, x.w);
    }
    for (int j = v0 + 4 * nvec + tid; j < hi; j += RANK_THREADS) visit(j, __ldcg(row + j));
    int tot;
    block_scan_incl(cand, s_warp, &tot);           // ends with a barrier: the histogram is complete
    if (ch == 0 && tid == 0 && tot) atomicAdd(&a.n_cand[b], (unsigned long long)tot);
    for (int j = tid; j < len; j += RANK_THREADS) {
      const int h = hist[j];
      if (h) atomicAdd(&a.cnt[base + c0 + j], h);
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(RANK_THREADS) k_rank_finish(RankArgs a) {
  __shared__ int s_warp[RANK_THREADS / 32];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int p0 = a.bt.ent_off[b], p1 = a.bt.ent_off[b + 1];
  const int n = a.n_rel[b];
  for (int i = p0 + tid; i < p1; i += RANK_THREADS) a.rank[i] = 0;
  __syncthreads();
  for (int c0 = 0; c0 < n; c0 += RANK_CHUNK) {
    const int len = min(RANK_CHUNK, n - c0);
    int carry = 0;
    for (int t0 = 0; t0 < len; t0 += RANK_THREADS) {
      const int t = t0 + tid;
      const int v = t < len ? a.cnt[p0 + c0 + t] : 0;
      int tot;
      const int r = carry + block_scan_incl(v, s_warp, &tot);
      if (t < len) a.rank[a.ent[p0 + c0 + t]] = r;
      carry += tot;
    }
  }
}

}  // namespace ocf
