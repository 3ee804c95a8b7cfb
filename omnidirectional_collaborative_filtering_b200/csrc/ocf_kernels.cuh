// Hand-written sm_100a kernels of the training / scoring hot path.
//
// Data layout in HBM (DESIGN.md section 3):
//   * rating store: CSR (rowptr i64, col i32, val f32)
//   * encoder kernel  Wenc  [k*N, HP]  (Keras layout, fan_out padded to a multiple of 128)
//   * decoder kernel  WdecT [N, HP]    (TRANSPOSED Keras layout: one contiguous row per
//     catalogue column, so the loss at an observed entry is one coalesced 4*HP-byte read)
//   * activations [B, HP] fp32
// Every catalogue-wide operation is therefore a gather of 4*HP-byte rows: row-centric kernels
// (one work item = a chunk of one batch row's ratings) for the activation-side products, and for
// the weight-side products a work list of (catalogue column, array) tasks - built from the batch
// by a counting sort (k_sort_*) - that a persistent kernel (k_row_update, one warp per task)
// turns into gradient rows fused with the optimizer update. All floating-point reductions run in
// a fixed order (no float atomics). The tensor-core scoring GEMM, the hidden-layer contractions and
// the top-k epilogue live in ocf_score_tc.cuh, ocf_gemm_tc.cuh and ocf_topk.cuh.
#pragma once

#include "ocf_common.cuh"

namespace ocf {

constexpr unsigned FULL = 0xffffffffu;

// ============================================================================================
// K1: CSR gather. Turns (row ids, keep flags) into the batch's rating tiles: column, value and
// a code byte saying which of the reference's dense arrays the rating is the live writer of.
// Replaces the per-rating Python loop of data_reader.py:122-170 / :226-268.
// One CTA per work item (a chunk of <= CH ratings of one row); reads and writes are contiguous.
// ============================================================================================
// RNG = true: the keep flag of a rating is derived here from the batch's slice of the NumPy
// MT19937 stream the generator workers left in the stream ring (draw d of the batch = its words 2d, 2d+1), compared with
// the row's cdf - what np.random.choice([0,1], n, p=[1-s, s]) returns (data_reader.py:130).
// The flags are also written back so a caller can read them.
template <bool RNG>
__global__ void __launch_bounds__(128)
k_gather_split(StoreDev s, BatchDev bt) {
  const BatchHdr hd = *bt.hdr;
  if ((int)blockIdx.x >= hd.n_items) return;
  const int pass_through = hd.pass_through;
  const int4 it = bt.items[blockIdx.x];
  const int b = it.x, start = it.y, len = it.z;
  const int row = bt.row_ids[b];
  const int64_t src0 = s.rowptr[row];
  const int p0 = bt.ent_off[b];
  const int d0 = RNG ? bt.draw_off[b] : 0;
  // the stream lives in a ring addressed by absolute position: word j of the batch's draws is ring word
  // (word_base + j) mod ring_words (a batch is shorter than the ring, so one conditional subtraction wraps)
  const uint32_t* W = RNG ? bt.words : nullptr;
  auto draw = [&](size_t d) -> double {
    uint32_t x0 = hd.word_base + 2u * (uint32_t)d, x1 = x0 + 1u;
    if (x0 >= hd.ring_words) x0 -= hd.ring_words;
    if (x1 >= hd.ring_words) x1 -= hd.ring_words;
    return mt_double(W[x0], W[x1]);
  };
  __shared__ double s_c0;
  if (RNG) {
    if (threadIdx.x == 0) {
      // the row's sparsity: draw (first row of the drawing unit + b) of np.random.uniform(lo, hi, size)
      // (data_reader.py:120), then the cdf np.random.choice builds from p = [1-s, s] (:130)
      const int r = hd.cdf_row0 + b;
      const double u = draw((size_t)r);
      const double keep = __dadd_rn(hd.rng_lo, __dmul_rn(hd.rng_range, u));   // random_uniform: lower + range * next_double
      const double q0 = __dsub_rn(1.0, keep);
      s_c0 = __ddiv_rn(q0, __dadd_rn(q0, keep));                             // cdf = cumsum(p) / cumsum(p)[-1]
    }
    __syncthreads();
  }
  const double c0 = RNG ? s_c0 : 0.0;
  auto flag_of = [&](int j) -> uint8_t {
    if (!RNG) return bt.flags[p0 + j];
    const size_t d = (size_t)(d0 + (s.orig_pos != nullptr ? s.orig_pos[src0 + j] : j));
    return draw(d) >= c0 ? 1 : 0;
  };
  for (int i = threadIdx.x; i < len; i += blockDim.x) {
    const int j = start + i;
    const int64_t src = src0 + j;
    const int p = p0 + j;
    const uint8_t f = flag_of(j);
    if (RNG) bt.flags_out[p] = f;
    bool in_live = f != 0;
    bool tg_live = (f == 0) || pass_through;
    bool obs_live = true;
    if (s.next_dup != nullptr) {
      int k = s.next_dup[src];
      while (k >= 0) {               // later ratings of the same column overwrite this one
        obs_live = false;
        const uint8_t fk = flag_of(k);
        if (fk != 0) in_live = false;
        if (fk == 0 || pass_through) tg_live = false;
        k = s.next_dup[src0 + k];
      }
    }
    bt.ent_col[p] = s.col[src];
    bt.ent_val[p] = s.val[src];
    bt.codes[p] = (uint8_t)((in_live ? CODE_IN : 0) | (obs_live ? CODE_OBS : 0) | (tg_live ? CODE_TGT : 0));
  }
}

// ============================================================================================
// NumPy's MT19937 stream on the device. A worker CTA owns a 624-word array. The recurrence
//   x[n] = x[n-227] ^ A(x[n-624], x[n-623])            (A = the "twist" of two neighbouring words)
// only reaches 227 words back through a plain XOR, so inside one regeneration the chain can be
// unrolled until it lands in the previous array: every new word is the XOR of at most three
// twists of OLD words and one old word,
//   i <  227 : new[i] = A(i) ^ old[i+397]
//   i <  454 : new[i] = A(i) ^ A(i-227) ^ old[i+170]
//   i <  623 : new[i] = A(i) ^ A(i-227) ^ A(i-454) ^ old[i-57]
//   i == 623 : new[623] = A(old[623], new[0]) ^ new[396]
// all 624 of them independent: two barriers per regeneration (twists evaluated once into shared
// memory), and every thread tempers and stores the word it produced. The tempered words leave
// through a small ring of slots in shared memory and TMA bulk stores (cp.async.bulk shared ->
// global): ordinary global stores inside the loop made every barrier wait for their
// acknowledgement; the bulk copies run in the async proxy and only a slot's reuse waits on them.
// One CTA tops out at ~0.84 G draws/s (one dependency chain). The stream is therefore produced in
// BLOCKS of a fixed number of regenerations by several worker CTAs side by side: worker j makes
// blocks j, j + M, j + 2M, ... and between two of its blocks JUMPS over the others' blocks with
// k_mt_jump_apply (GF(2) polynomial jump-ahead, ocf_mtjump.h). The result is the sequential
// stream, bit for bit. Consumers (k_gather_split) address the ring by absolute stream position.
// ============================================================================================
__device__ __forceinline__ uint32_t mt_twist(uint32_t cur, uint32_t nxt, uint32_t far) {
  const uint32_t y = (cur & 0x80000000u) | (nxt & 0x7fffffffu);
  return far ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
}
__device__ __forceinline__ uint32_t mt_temper(uint32_t y) {
  y ^= y >> 11;
  y ^= (y << 7) & 0x9d2c5680u;
  y ^= (y << 15) & 0xefc60000u;
  y ^= y >> 18;
  return y;
}

__device__ __forceinline__ uint32_t mt_a(uint32_t cur, uint32_t nxt) {
  const uint32_t y = (cur & 0x80000000u) | (nxt & 0x7fffffffu);
  return (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
}

constexpr int MT_THREADS = 640;            // one word of a regeneration per thread (624 active)
constexpr int MT_RING = 4;                 // regenerations in flight towards HBM
constexpr int MT_SEQ_REGENS = 33;          // arrays a jump reads: 33 * 624 >= 19937 + 624 words of the worker's own sequence

// One word of the new array from twists of the old one (see the derivation above). own = tw[i].
__device__ __forceinline__ uint32_t mt_new_word(int i, uint32_t own, const uint32_t* __restrict__ o, const uint32_t* __restrict__ tw) {
  if (i < 227) return own ^ o[i + 397];
  if (i < 454) return own ^ tw[i - 227] ^ o[i + 170];
  if (i < 623) return own ^ tw[i - 227] ^ tw[i - 454] ^ o[i - 57];
  return mt_a(o[623], tw[0] ^ o[397]) ^ (tw[396] ^ tw[169] ^ o[566]);
}

// A block of the stream: `n_regen` regenerations continuing the 624-word array `state` (left at the array after
// the last one). TEMPER: the tempered words (what NumPy hands out) go to the ring buffer `ring` of `ring_words`
// words at word offset `off0` (a multiple of 4, every regeneration 16-byte aligned; a regeneration never straddles
// the ring's end because ring_words is a multiple of 624) through shared-memory slots and TMA bulk stores. Without
// TEMPER the raw arrays are appended to `ring` from off0 (the sequence a jump correlates with its polynomial).
// One launch per block and two per jump: every launch costs the host ~3 us, and a rank of an 8-GPU run makes
// ~10 blocks per step (profiles/r02: 0.29 ms of API calls per step with the 8-call version of block + jump).
// state[626..629]: SM cycles and nanoseconds of the launch (ocf_rng_last_timing).
template <bool TEMPER>
__global__ void __launch_bounds__(MT_THREADS)
k_mt_block(uint32_t* __restrict__ state, int n_regen, uint32_t* __restrict__ ring, uint32_t ring_words, uint32_t off0,
           const uint32_t* __restrict__ src = nullptr, uint32_t* __restrict__ clear = nullptr) {
  __shared__ __align__(16) uint32_t mt[2][624];
  __shared__ __align__(16) uint32_t tw[624];
  __shared__ __align__(16) uint32_t slots[MT_RING][624];
  const int tid = threadIdx.x;
  const long long clk0 = clock64();
  unsigned long long ns0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns0));
  // src (a jump's sequence pass): start from `src` and leave it alone - its raw words open the sequence at
  // ring[off0 - 624 ..), nothing is written back; `clear` (the jump's output array) is zeroed on the way out.
  for (int i = tid; i < 624; i += blockDim.x) {
    const uint32_t v = src != nullptr ? src[i] : state[i];
    mt[0][i] = v;
    if (src != nullptr) ring[off0 - 624u + i] = v;
  }
  int cur = 0;
  __syncthreads();
  uint32_t off = off0;
  // A single CTA is bound by the latency of each thread's dependent instruction chain between the two barriers
  // (measured: fewer, busier threads are slower), so every word gets its own thread and the shortest chain.
  const int i = tid;
  const bool active = i < 624;
  for (int g = 0; g < n_regen; ++g) {
    const uint32_t* o = mt[cur];
    uint32_t* n = mt[cur ^ 1];
    uint32_t* slot = slots[g % MT_RING];
    uint32_t own = 0u;
    if (i < 623) { own = mt_a(o[i], o[i + 1]); tw[i] = own; }     // word 623 has no plain twist (it needs new[0])
    if (tid == 0 && g >= MT_RING)                                  // the bulk store that last read this slot has its data
      asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(MT_RING - 1) : "memory");
    __syncthreads();
    if (active) {
      const uint32_t v = mt_new_word(i, own, o, tw);
      n[i] = v;
      slot[i] = TEMPER ? mt_temper(v) : v;
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
      asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                   ::"l"(ring + off), "r"((uint32_t)__cvta_generic_to_shared(slot)), "r"(624u * 4u) : "memory");
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
    off += 624u;
    if (off >= ring_words) off -= ring_words;
    cur ^= 1;
  }
  if (tid == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  __syncthreads();
  if (clear != nullptr) for (int k = tid; k < 624; k += blockDim.x) clear[k] = 0u;
  if (src != nullptr) return;
  for (int k = tid; k < 624; k += blockDim.x) state[k] = mt[cur][k];
  if (tid == 0) {
    unsigned long long ns1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns1));
    const unsigned long long cyc = (unsigned long long)(clock64() - clk0), ns = ns1 - ns0;
    state[626] = (uint32_t)cyc; state[627] = (uint32_t)(cyc >> 32);
    state[628] = (uint32_t)ns; state[629] = (uint32_t)(ns >> 32);
  }
}

// Jump of a worker's array by J words, J fixed by the polynomial g = x^J mod phi (ocf_mtjump.h):
//   out[k] = XOR over the set bits i of g of seq[i + k],   seq = the worker's own untempered sequence
// (seq[0..623] = its current array, then MT_SEQ_REGENS - 1 further arrays from k_mt_block<false>). CTA c takes bits
// [624 c, 624 c + 624) of g with its slice of the sequence staged in shared memory; the partial arrays are combined
// with integer XOR atomics (order-independent, so the result is exact and reproducible). out must be zeroed.
constexpr int MT_JUMP_CTAS = 32;           // 32 * 624 = 19968 >= 19937 polynomial bits

__global__ void __launch_bounds__(MT_THREADS)
k_mt_jump_apply(const uint32_t* __restrict__ seq, const uint32_t* __restrict__ poly, uint32_t* __restrict__ out) {
  __shared__ uint32_t s_seq[1248];
  __shared__ uint32_t s_poly[20];            // 624 bits from bit0 (bit0 % 32 is 0 or 16) lie in exactly 20 words
  const int tid = threadIdx.x;
  const int bit0 = blockIdx.x * 624;
  for (int k = tid; k < 1248; k += blockDim.x) s_seq[k] = seq[bit0 + k];
  if (tid < 20) s_poly[tid] = (bit0 >> 5) + tid < 624 ? poly[(bit0 >> 5) + tid] : 0u;
  __syncthreads();
  if (tid >= 624) return;
  uint32_t acc = 0u;
  const int sh = bit0 & 31;
  for (int b = 0; b < 624; ++b) {
    const int pos = sh + b;
    if ((s_poly[pos >> 5] >> (pos & 31)) & 1u) acc ^= s_seq[b + tid];
  }
  if (acc) atomicXor(&out[tid], acc);
}

// Fixed-split valid/test batches: a batch row is the input store's row followed by the target
// store's row. in_overlap[e] != 0 marks input ratings whose column is also a target of the row
// (the missing-data mask is then carried by the target entry only).
__global__ void __launch_bounds__(128)
k_gather_fixed(StoreDev sin, StoreDev stg, const uint8_t* __restrict__ in_overlap, BatchDev bt) {
  if ((int)blockIdx.x >= bt.hdr->n_items) return;
  const int4 it = bt.items[blockIdx.x];
  const int b = it.x, start = it.y, len = it.z;
  const int row = bt.row_ids[b];
  const int nin = bt.in_len[b];
  const int64_t in0 = sin.rowptr[row], tg0 = stg.rowptr[row];
  const int p0 = bt.ent_off[b];
  for (int i = threadIdx.x; i < len; i += blockDim.x) {
    const int j = start + i;
    const int p = p0 + j;
    int c; float v; uint8_t code;
    if (j < nin) {
      const int64_t src = in0 + j;
      c = sin.col[src]; v = sin.val[src];
      const bool live = sin.next_dup == nullptr || sin.next_dup[src] < 0;
      const bool also_target = in_overlap != nullptr && in_overlap[src] != 0;
      code = live ? (uint8_t)(CODE_IN | (also_target ? 0 : CODE_OBS)) : 0;
    } else {
      const int64_t src = tg0 + (j - nin);
      c = stg.col[src]; v = stg.val[src];
      const bool live = stg.next_dup == nullptr || stg.next_dup[src] < 0;
      code = live ? (uint8_t)(CODE_TGT | CODE_OBS) : 0;
    }
    bt.ent_col[p] = c; bt.ent_val[p] = v; bt.codes[p] = code;
  }
}

// The scatter half of K1: the dense float64 [B, N] arrays of data_reader.py:191-200, for parity
// tests and callers that want Keras-style feeds. `out` must be zeroed.
__global__ void k_densify(BatchDev bt, int which, double aux_val, int n_cols, double* __restrict__ out) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= bt.n_entries) return;
  // batch row of entry p: binary search in ent_off
  int lo = 0, hi = bt.B;
  while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (bt.ent_off[mid] <= p) lo = mid; else hi = mid; }
  const uint8_t code = bt.codes[p];
  const double v = (double)bt.ent_val[p];
  double w; bool on;
  switch (which) {
    case 0: on = code & CODE_IN; w = v; break;
    case 1: on = code & CODE_IN; w = aux_val; break;
    case 2: on = code & CODE_TGT; w = aux_val; break;
    case 3: on = code & CODE_TGT; w = v; break;
    default: on = code & CODE_OBS; w = aux_val; break;
  }
  if (on) out[(size_t)lo * n_cols + bt.ent_col[p]] = w;
}

// ============================================================================================
// z + bias -> activation -> inverted dropout (model.py:66-73). Padded units are forced to 0.
// a_out: activation before dropout (needed for the derivative), h_out: what the next layer sees,
// dscale: 0 or 1/(1-p) per element (null when dropout is off). The dropout counter (step) and key
// come from the model's device-resident StepDev.
// ============================================================================================
struct ActArgs {
  const float4* bias; int B; int H; int hp4; int act;
  float4* a_out; float4* h_out; float4* dscale;
  float p_drop; const StepDev* st; uint32_t layer; int row0;
};

__device__ __forceinline__ void bias_act_elem(const ActArgs& g, int idx, const float4 z) {
  const int b = idx / g.hp4, u4 = idx - b * g.hp4;
  const float4 bb = g.bias[u4];
  float a[4] = {z.x + bb.x, z.y + bb.y, z.z + bb.z, z.w + bb.w};
#pragma unroll
  for (int k = 0; k < 4; ++k) a[k] = (u4 * 4 + k < g.H) ? act_fwd(g.act, a[k]) : 0.f;
  g.a_out[idx] = make_float4(a[0], a[1], a[2], a[3]);
  if (g.dscale != nullptr) {
    const uint32_t step = g.st->step;
    const uint2 key = make_uint2(g.st->seed_lo, g.st->seed_hi);
    const uint4 r = philox4x32_10(make_uint4((uint32_t)u4, (uint32_t)(b + g.row0), g.layer, step), key);
    const uint32_t thresh = (uint32_t)floor((double)g.p_drop * 16777216.0);
    const float inv = 1.0f / (1.0f - g.p_drop);
    const uint32_t rr[4] = {r.x, r.y, r.z, r.w};
    float sc[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) { sc[k] = ((rr[k] >> 8) >= thresh) ? inv : 0.f; a[k] *= sc[k]; }
    g.dscale[idx] = make_float4(sc[0], sc[1], sc[2], sc[3]);
  }
  g.h_out[idx] = make_float4(a[0], a[1], a[2], a[3]);
}

__global__ void __launch_bounds__(256)
k_bias_act(const float4* __restrict__ zsum, ActArgs g) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= g.B * g.hp4) return;
  bias_act_elem(g, idx, zsum[idx]);
}

// ============================================================================================
// Row tail of the row-centric kernels (K2, K3). A batch row's ratings are spread over work items
// (one CTA each); the row's result is the sum of its items' partial rows. Instead of a separate
// reduction kernel, the CTAs of a row count their arrivals and the LAST one to arrive sums the
// partials - always in item order, so the result does not depend on which CTA that is. Rows with
// more than TAIL_FAN items reduce in two levels (groups of TAIL_FAN consecutive items, then the
// groups), which bounds the serial part of a heavy row (hundreds of items) to two short sums.
// Counters reset themselves; every batch row has at least one item (an empty row has one item of
// length 0), so every row gets its tail.
// ============================================================================================
constexpr int TAIL_FAN = 16;

struct TailBuf {
  int* tick_grp;      // [max_items] arrivals of a group, indexed by the group's first item
  int* tick_row;      // [max_rows]  arrivals of a row's groups
  float4* G;          // [max_items, hp4] group sums, indexed by the group's first item
  float* Gs;          // [max_items, ROWSTAT_W] group sums of the loss statistics
};

// sum of `count` partial rows P[(first + k * step) * hp4 + u], k = 0..count-1, fixed order, 4 accumulators
__device__ __forceinline__ float4 tail_sum4(const float4* P, int first, int step, int count, int hp4, int u) {
  float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0, a2 = a0, a3 = a0;
  int k = 0;
  for (; k + 8 <= count; k += 8) {
    float4 p[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) p[q] = __ldcg(P + (size_t)(first + (k + q) * step) * hp4 + u);
#pragma unroll
    for (int q = 0; q < 8; q += 4) {
      a0.x += p[q].x; a0.y += p[q].y; a0.z += p[q].z; a0.w += p[q].w;
      a1.x += p[q + 1].x; a1.y += p[q + 1].y; a1.z += p[q + 1].z; a1.w += p[q + 1].w;
      a2.x += p[q + 2].x; a2.y += p[q + 2].y; a2.z += p[q + 2].z; a2.w += p[q + 2].w;
      a3.x += p[q + 3].x; a3.y += p[q + 3].y; a3.z += p[q + 3].z; a3.w += p[q + 3].w;
    }
  }
  for (; k < count; ++k) {
    const float4 p = __ldcg(P + (size_t)(first + k * step) * hp4 + u);
    float4& a = (k & 3) == 0 ? a0 : ((k & 3) == 1 ? a1 : ((k & 3) == 2 ? a2 : a3));
    a.x += p.x; a.y += p.y; a.z += p.z; a.w += p.w;
  }
  return make_float4((a0.x + a1.x) + (a2.x + a3.x), (a0.y + a1.y) + (a2.y + a3.y),
                     (a0.z + a1.z) + (a2.z + a3.z), (a0.w + a1.w) + (a2.w + a3.w));
}

// Runs at the end of a row-centric CTA (all threads, after the CTA's own partial row / statistics are
// in global memory). `finish(u, sum)` receives the row's summed float4 column u (u < hp4; hp4 = 0: no
// row data), `finish_stat(k, sum)` the row's summed statistic k when `stats` is given.
template <typename F, typename FS>
__device__ __forceinline__ void row_tail(const BatchDev& bt, int item, int b, const float4* P, int hp4,
                                         const float* stats, const TailBuf& tb, F&& finish, FS&& finish_stat) {
  __shared__ int s_last;
  const int i0 = bt.item_ptr[b], i1 = bt.item_ptr[b + 1];
  const int n = i1 - i0;
  const int nthreads = blockDim.x;
  if (n == 1) {                                   // the CTA's own partial is the row (bar.sync orders the CTA's global writes)
    __syncthreads();
    for (int u = threadIdx.x; u < hp4; u += nthreads) finish(u, P[(size_t)item * hp4 + u]);
    if (stats != nullptr && threadIdx.x < ROWSTAT_W) finish_stat((int)threadIdx.x, stats[(size_t)item * ROWSTAT_W + threadIdx.x]);
    return;
  }
  const int g_first = i0 + (item - i0) / TAIL_FAN * TAIL_FAN;
  const int g_count = min(TAIL_FAN, i1 - g_first);
  const int n_groups = (n + TAIL_FAN - 1) / TAIL_FAN;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const int t = atomicAdd(&tb.tick_grp[g_first], 1);
    s_last = t == g_count - 1;
    if (s_last) tb.tick_grp[g_first] = 0;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  if (n_groups == 1) {
    for (int u = threadIdx.x; u < hp4; u += nthreads) finish(u, tail_sum4(P, g_first, 1, g_count, hp4, u));
    if (stats != nullptr && threadIdx.x < ROWSTAT_W) {
      float s = 0.f;
      for (int k = 0; k < g_count; ++k) s += __ldcg(stats + (size_t)(g_first + k) * ROWSTAT_W + threadIdx.x);
      finish_stat((int)threadIdx.x, s);
    }
    return;
  }
  for (int u = threadIdx.x; u < hp4; u += nthreads) tb.G[(size_t)g_first * hp4 + u] = tail_sum4(P, g_first, 1, g_count, hp4, u);
  if (stats != nullptr && threadIdx.x < ROWSTAT_W) {
    float s = 0.f;
    for (int k = 0; k < g_count; ++k) s += __ldcg(stats + (size_t)(g_first + k) * ROWSTAT_W + threadIdx.x);
    tb.Gs[(size_t)g_first * ROWSTAT_W + threadIdx.x] = s;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const int t = atomicAdd(&tb.tick_row[b], 1);
    s_last = t == n_groups - 1;
    if (s_last) tb.tick_row[b] = 0;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  for (int u = threadIdx.x; u < hp4; u += nthreads) finish(u, tail_sum4(tb.G, i0, TAIL_FAN, n_groups, hp4, u));
  if (stats != nullptr && threadIdx.x < ROWSTAT_W) {
    float s = 0.f;
    for (int k = 0; k < n_groups; ++k) s += __ldcg(tb.Gs + (size_t)(i0 + k * TAIL_FAN) * ROWSTAT_W + threadIdx.x);
    finish_stat((int)threadIdx.x, s);
  }
}

// ============================================================================================
// K2: encoder, sparse-row x dense Wenc (SpMM). Work item = chunk of one batch row; the 4 warps of
// the CTA split the chunk's ratings, each warp accumulates full HP-wide rows (NV float4 per
// lane, 512-byte coalesced segments), then the warps are summed in a fixed order.
// x0 = [data | aux | second] (model.py:47-56) is never formed: block k of the concatenation is
// rows [k*N, (k+1)*N) of Wenc, selected by the entry's code bits.
// The row's last CTA (row_tail) sums the row and either stores the pre-activation z (a column shard
// all-reduces it first) or applies bias + activation + dropout right there (fuse_act).
// ============================================================================================
// Ties whatever is computed from `dep` afterwards to every 16-byte load of the row: dep += 0 * (one component of each
// load), which IEEE arithmetic cannot fold away and which stays 0 for finite weights. ptxas otherwise interleaves the
// FMAs of row q with the loads of row q + 1 to save registers (cuobjdump: 4 LDG, 7 FFMA, 1 LDG, 9 FFMA, ...), and the
// warp then waits for row q before row q + 1 is even requested: one row in flight instead of RIF.
template <int NV>
__device__ __forceinline__ void depend_on_row(float& dep, const float4 (&w)[NV]) {
#pragma unroll
  for (int v = 0; v < NV; ++v) dep = fmaf(0.f, w[v].x, dep);
}

template <int NV>
__global__ void __launch_bounds__(128)
k_enc_fwd(BatchDev bt, const float* __restrict__ Wenc, int n_cols, int nblk, int3 bits,
          float4* __restrict__ P, TailBuf tb, float4* __restrict__ z_out, int fuse_act, ActArgs act) {
  pdl_trigger();
  pdl_wait();
  constexpr int HP = NV * 128;
  constexpr int RIF = 2;                    // weight rows in flight per warp and round (3 and 4 cost more occupancy than they add: 46-47 vs 42.6 us, ML-10M shape)
  __shared__ float4 red[4][HP / 4];
  __shared__ int2 s_list[128 * 3];          // (weight row, coefficient bits) of the row loads of 128 entries
  __shared__ int s_cnt[3][4];
  // header and item are read together (the launch never exceeds the item array's capacity), and the item carries the
  // absolute position of its first entry: the chain to the first weight row is header/item -> entries -> rows
  const int4 it = bt.items[blockIdx.x];
  const int n_items = bt.hdr->n_items;
  const float aux_val = bt.hdr->aux_value;
  if ((int)blockIdx.x >= n_items) return;
  const int len = it.z;
  const int p0 = it.w;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float4 acc[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);

  // The chunk's (entry, input block) pairs that really load a weight row are compacted into one list in shared
  // memory (entry order within a block, blocks in order), and the four warps deal that list in pairs: every warp
  // gets the same number of row loads whatever the keep flags look like. (Dealing the ENTRIES to the warps left a
  // third of the warp time waiting at the barrier for the warp that drew the most inputs.)
  for (int tile = 0; tile < len; tile += 128) {
    const int i = tile + (int)threadIdx.x;
    int c = 0, code = 0; float val = 0.f;
    if (i < len) { c = bt.ent_col[p0 + i]; val = bt.ent_val[p0 + i]; code = bt.codes[p0 + i]; }
    unsigned bal[3];
#pragma unroll
    for (int blk = 0; blk < 3; ++blk) {
      const int bit = blk == 0 ? bits.x : (blk == 1 ? bits.y : bits.z);
      bal[blk] = blk < nblk ? __ballot_sync(FULL, (code & bit) != 0) : 0u;
      if (lane == 0) s_cnt[blk][warp] = __popc(bal[blk]);
    }
    __syncthreads();
    int total = 0;
#pragma unroll
    for (int blk = 0; blk < 3; ++blk) {
      int mine = total;
#pragma unroll
      for (int w2 = 0; w2 < 4; ++w2) { const int n = s_cnt[blk][w2]; if (w2 < warp) mine += n; total += n; }
      if ((bal[blk] >> lane) & 1u)
        s_list[mine + __popc(bal[blk] & ((1u << lane) - 1u))] = make_int2(blk * n_cols + c, __float_as_int(blk == 0 ? val : aux_val));
    }
    __syncthreads();
    // RIF rows in flight per warp and round: the kernel is bound by (rounds per warp) x (latency of a round)
    // (a round past the end of the list re-reads its last row, x 0)
    for (int j = warp * RIF; j < total; j += 4 * RIF) {
      float f[RIF];
      const float* r[RIF];
#pragma unroll
      for (int q = 0; q < RIF; ++q) {
        const int2 e = s_list[min(j + q, total - 1)];
        f[q] = j + q < total ? __int_as_float(e.y) : 0.f;
        r[q] = Wenc + (size_t)e.x * HP + lane * 4;
      }
      float4 w[RIF][NV];
#pragma unroll
      for (int q = 0; q < RIF; ++q)
#pragma unroll
        for (int v = 0; v < NV; ++v) w[q][v] = ldg4(r[q] + v * 128);
      float dep = 0.f;
      if (NV <= 4) {                           // wide rows: two of them already fill the register file
#pragma unroll
        for (int q = 0; q < RIF; ++q) depend_on_row<NV>(dep, w[q]);
      }
#pragma unroll
      for (int q = 0; q < RIF; ++q) {
        const float fq = f[q] + dep;           // + 0, but only once every row of the round has landed
#pragma unroll
        for (int v = 0; v < NV; ++v) fma4(acc[v], fq, w[q][v]);
      }
    }
    if (tile + 128 < len) __syncthreads();          // the list is rebuilt for the next 128 entries
  }
#pragma unroll
  for (int v = 0; v < NV; ++v) red[warp][v * 32 + lane] = acc[v];
  __syncthreads();
  for (int u = threadIdx.x; u < HP / 4; u += 128) {
    float4 s = red[0][u];
    const float4 a = red[1][u], b2 = red[2][u], c2 = red[3][u];
    s.x = ((s.x + a.x) + b2.x) + c2.x; s.y = ((s.y + a.y) + b2.y) + c2.y;
    s.z = ((s.z + a.z) + b2.z) + c2.z; s.w = ((s.w + a.w) + b2.w) + c2.w;
    P[(size_t)blockIdx.x * (HP / 4) + u] = s;
  }
  const int b = it.x;
  row_tail(bt, (int)blockIdx.x, b, P, HP / 4, nullptr, tb,
           [&](int u, const float4 z) {
             const int idx = b * (HP / 4) + u;
             if (fuse_act) bias_act_elem(act, idx, z); else z_out[idx] = z;
           },
           [&](int, float) {});
}

// ============================================================================================
// K3: decoder at the observed target entries (SDDMM) fused with bias, output mask, masked
// loss, metrics and the loss gradient; accumulates dL/dh on the fly. The dense [B, N]
// reconstruction (model.py:82-86) is never formed.
//   full = h . WdecT[c] + b[c];  y = m * full (m = aux_var_value);  e = y - t
//   dL/dfull = m * 2e/(B N)   (mean_squared_error)   or   m * sign(e)/(B N)   (mean_absolute_error)
// The row's last CTA (row_tail) leaves the row's loss statistics in rowstats[b] and, when training,
// dL/dh of the row in dh_out[b].
// ============================================================================================
// With `fz.dz` set (an unsharded model: dL/dh of a row is complete on this device) the row's last CTA goes one step
// further and leaves dz = dL/dh * dropout scale * act'(a) of the top hidden layer: the first kernel of the backward
// pass (k_dz_bias) then only sums columns for the bias, off the step's critical path.
struct DzFuse { const float4* a; const float4* dscale; float4* dz; int act; };

template <int NV, bool TRAIN>
__global__ void __launch_bounds__(128, NV <= 4 ? 6 : 3)
k_dec_fwd(BatchDev bt, const float* __restrict__ WdecT, const float* __restrict__ bdec,
          const float* __restrict__ h, float gscale, int loss_kind,
          float* __restrict__ dy, float4* __restrict__ P2, float* __restrict__ itemstats,
          float* __restrict__ dense_out, int n_cols, TailBuf tb, float4* __restrict__ dh_out, float* __restrict__ rowstats, DzFuse fz) {
  pdl_trigger();
  pdl_wait();
  constexpr int HP = NV * 128;
  __shared__ float4 red[TRAIN ? 4 : 1][HP / 4];
  __shared__ float sred[4][3];
  __shared__ int2 s_list[128];              // (column, entry) of the target entries of 128 entries
  __shared__ float s_t[128];
  __shared__ int s_cnt[4];
  // the batch row's activations sit in shared memory, not in NV float4 registers per lane: the kernel is bound by how
  // many warps (rows in flight) an SM holds, and 16 registers less is one more resident CTA per SM
  __shared__ float4 s_h[HP / 4];
  const int4 it = bt.items[blockIdx.x];     // header and item together, item.w = first entry (see k_enc_fwd)
  const int n_items = bt.hdr->n_items;
  const float aux_val = bt.hdr->aux_value;
  if ((int)blockIdx.x >= n_items) return;
  const int b = it.x, len = it.z;
  const int p0 = it.w;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float4 dh[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v) dh[v] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int u = threadIdx.x; u < HP / 4; u += 128) s_h[u] = ldg4(h + (size_t)b * HP + u * 4);   // published by the tile loop's first barrier
  float sse = 0.f, sae = 0.f, cnt = 0.f;

  // target entries compacted into a list in shared memory, dealt to the four warps in pairs (see k_enc_fwd)
  for (int tile = 0; tile < len; tile += 128) {
    const int i = tile + (int)threadIdx.x;
    int c = 0, code = 0; float t = 0.f;
    if (i < len) { c = bt.ent_col[p0 + i]; t = bt.ent_val[p0 + i]; code = bt.codes[p0 + i]; }
    const bool tgt = (code & CODE_TGT) != 0;
    if (TRAIN && i < len && !tgt) dy[p0 + i] = 0.f;
    const unsigned bal = __ballot_sync(FULL, tgt);
    if (lane == 0) s_cnt[warp] = __popc(bal);
    __syncthreads();
    int mine = 0, total = 0;
#pragma unroll
    for (int w2 = 0; w2 < 4; ++w2) { const int n = s_cnt[w2]; if (w2 < warp) mine += n; total += n; }
    if (tgt) { const int pos = mine + __popc(bal & ((1u << lane) - 1u)); s_list[pos] = make_int2(c, i); s_t[pos] = t; }
    __syncthreads();
    for (int j = warp * 2; j < total; j += 8) {
      const bool two = j + 1 < total;
      const int2 e0 = s_list[j], e1 = s_list[two ? j + 1 : j];
      const int c0 = e0.x, c1 = e1.x;
      const float t0 = s_t[j], t1 = s_t[two ? j + 1 : j];
      const float* r0 = WdecT + (size_t)c0 * HP + lane * 4;
      const float* r1 = WdecT + (size_t)c1 * HP + lane * 4;
      float4 w0[NV], w1[NV];
#pragma unroll
      for (int v = 0; v < NV; ++v) { w0[v] = ldg4(r0 + v * 128); w1[v] = ldg4(r1 + v * 128); }
      const float bias0 = __ldg(bdec + c0), bias1 = __ldg(bdec + c1);
      float dep = 0.f;
      if (NV <= 4) { depend_on_row<NV>(dep, w0); depend_on_row<NV>(dep, w1); }      // both rows requested before either is used (see k_enc_fwd)
      float d0 = dep, d1 = dep;
#pragma unroll
      for (int v = 0; v < NV; ++v) { const float4 hv = s_h[v * 32 + lane]; d0 = dot4(w0[v], hv, d0); d1 = dot4(w1[v], hv, d1); }
      d0 = warp_sum(d0); d1 = warp_sum(d1);
      {
        const float y = aux_val * (d0 + bias0), e = y - t0;
        sse = fmaf(e, e, sse); sae += fabsf(e); cnt += ((t0 + y) != 0.f) ? 1.f : 0.f;
        if (dense_out != nullptr && lane == 0) dense_out[(size_t)b * n_cols + c0] = y;
        if (TRAIN) {
          const float ge = loss_kind == OCF_LOSS_MSE ? gscale * e : gscale * (float)((e > 0.f) - (e < 0.f));
          const float dyv = aux_val * ge;
          if (lane == 0) dy[p0 + e0.y] = dyv;
#pragma unroll
          for (int v = 0; v < NV; ++v) fma4(dh[v], dyv, w0[v]);
        }
      }
      if (two) {
        const float y = aux_val * (d1 + bias1), e = y - t1;
        sse = fmaf(e, e, sse); sae += fabsf(e); cnt += ((t1 + y) != 0.f) ? 1.f : 0.f;
        if (dense_out != nullptr && lane == 0) dense_out[(size_t)b * n_cols + c1] = y;
        if (TRAIN) {
          const float ge = loss_kind == OCF_LOSS_MSE ? gscale * e : gscale * (float)((e > 0.f) - (e < 0.f));
          const float dyv = aux_val * ge;
          if (lane == 0) dy[p0 + e1.y] = dyv;
#pragma unroll
          for (int v = 0; v < NV; ++v) fma4(dh[v], dyv, w1[v]);
        }
      }
    }
    if (tile + 128 < len) __syncthreads();
  }
  if (lane == 0) { sred[warp][0] = sse; sred[warp][1] = sae; sred[warp][2] = cnt; }
  if (TRAIN) {
#pragma unroll
    for (int v = 0; v < NV; ++v) red[warp][v * 32 + lane] = dh[v];
  }
  __syncthreads();
  if (TRAIN) {
    for (int u = threadIdx.x; u < HP / 4; u += 128) {
      float4 s = red[0][u];
      const float4 a = red[1][u], b2 = red[2][u], c2 = red[3][u];
      s.x = ((s.x + a.x) + b2.x) + c2.x; s.y = ((s.y + a.y) + b2.y) + c2.y;
      s.z = ((s.z + a.z) + b2.z) + c2.z; s.w = ((s.w + a.w) + b2.w) + c2.w;
      P2[(size_t)blockIdx.x * (HP / 4) + u] = s;
    }
  }
  if (threadIdx.x < 3)
    itemstats[(size_t)blockIdx.x * ROWSTAT_W + threadIdx.x] =
        ((sred[0][threadIdx.x] + sred[1][threadIdx.x]) + sred[2][threadIdx.x]) + sred[3][threadIdx.x];
  if (threadIdx.x == 3) itemstats[(size_t)blockIdx.x * ROWSTAT_W + 3] = 0.f;
  row_tail(bt, (int)blockIdx.x, b, P2, TRAIN ? HP / 4 : 0, itemstats, tb,
           [&](int u, const float4 s) {
             const size_t idx = (size_t)b * (HP / 4) + u;
             if (fz.dz == nullptr) { dh_out[idx] = s; return; }
             float4 d = s;                     // the arithmetic of k_dz_bias, element for element
             if (fz.dscale != nullptr) { const float4 sc = fz.dscale[idx]; d.x *= sc.x; d.y *= sc.y; d.z *= sc.z; d.w *= sc.w; }
             const float4 av = fz.a[idx];
             d.x *= act_bwd(fz.act, av.x); d.y *= act_bwd(fz.act, av.y); d.z *= act_bwd(fz.act, av.z); d.w *= act_bwd(fz.act, av.w);
             fz.dz[idx] = d;
           },
           [&](int k, float s) { rowstats[(size_t)b * ROWSTAT_W + k] = s; });
}

// dz = dh * dropout scale * act'(a) for one hidden layer, the bias gradient (column sum over the
// batch) and the bias update. One CTA per 32 hidden units; its 32 warps deal the batch rows
// round-robin and their partial column sums are added in warp order. The launch may carry one
// CTA more than there are unit groups: it writes the step's metric record (saves a launch on the
// critical path of a training step).
// dh_is_dz: the input already is dz (left by K3's DzFuse or by the backward product's GEPI_DZ epilogue).
constexpr int LOG_CAP = 4096;             // steps the metric log holds
constexpr int LOG_W = OCF_N_METRICS;

struct MetricArgs {            // the step's metric record, written by one extra CTA of k_dz_bias (null log: none)
  const float* rowstats; int rows; float rows_total; float n_cols_total; float rating_range; int loss_kind;
  const float* regparts; int n_reg; float l2;
  float* log;                  // [LOG_CAP, LOG_W] page-locked host memory, written straight from the kernel
  StepDev* st;                 // the record goes to slot st->log_slot, which then advances
  int advance_step;            // training: the dropout counter advances too
};
__device__ void metrics_record(const MetricArgs& a, int lane);

__global__ void __launch_bounds__(1024)
k_dz_bias(const float* __restrict__ dh, const float* __restrict__ a, const float* __restrict__ dscale,
          int B, int HP, int act, int dh_is_dz, float* __restrict__ dz, float* __restrict__ bias,
          float* __restrict__ s1, float* __restrict__ s2, OptDev o, int trainable, float* __restrict__ gbias,
          MetricArgs met) {
  pdl_trigger();
  pdl_wait();
  __shared__ float part[32][32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (blockIdx.x * 32 >= HP) {           // the extra CTA: metrics of the step (train.py:102-121)
    if (warp == 0 && met.log != nullptr) metrics_record(met, lane);
    return;
  }
  const int u = blockIdx.x * 32 + lane;
  float g = 0.f;
  if (u < HP) {
    for (int b = warp; b < B; b += 32) {
      const size_t k = (size_t)b * HP + u;
      float d = dh[k];
      if (!dh_is_dz) {
        if (dscale != nullptr) d *= dscale[k];
        d *= act_bwd(act, a[k]);
        dz[k] = d;
      }
      g += d;
    }
  }
  part[warp][lane] = g;
  __syncthreads();
  if (warp == 0 && u < HP && trainable) {
    g = part[0][lane];
#pragma unroll
    for (int w = 1; w < 32; ++w) g += part[w][lane];
    if (gbias != nullptr) { gbias[u] = g; return; }   // row-parallel mode: the gradient is reduced over ranks first
    o.l2x2 = 0.f;                     // Keras regularises kernels only (model.py:66,82)
    float w = bias[u], t1 = s1 ? s1[u] : 0.f, t2 = s2 ? s2[u] : 0.f;
    opt_apply(o, o.st->lr, g, w, t1, t2);
    bias[u] = w;
    if (s1) s1[u] = t1;
    if (s2) s2[u] = t2;
  }
}

// ============================================================================================
// K4: weight-side products fused with the optimizer update: a work list, then the update.
//
// K4a (k_sort_*) groups the batch's own ratings by catalogue column with a counting sort over the
// ~10^5 gathered entries:
//   count   per entry: the column's count of matched batch rows, the OR of its code bits (int atomics) and
//           bit `batch row` of the column's row of the presence bitmap [n_cols][W words]
//   alloc   per COLUMN (a coalesced sweep over the count array): a touched column reserves its segment of
//           the match list and its update tasks; one atomic per warp and counter (warp-aggregated), and
//           the tasks come out in column order inside a warp: neighbouring tasks touch neighbouring
//           weight rows. One task per weight row that must change:
//             array 0      decoder row  WdecT[c,:]  (+ b_dec[c])   needs a target entry
//             array 1+blk  encoder row  Wenc[blk*N+c,:]            needs an entry with the block's bit
//           With a dense rule (RMSprop / Adam / L2) every row changes: alloc also records each touched
//           column's segment and the update enumerates all (column, array) pairs.
//   place   per entry: rank inside its column = popcount of the lower batch rows present, so a column's
//           matches are ordered by batch row whatever order the atomics ran in: the gradient sums of K4b
//           keep a fixed order (bit-reproducible steps)
// A match record is one (batch row, column) cell: (batch row | code << 16, value, entry index). When a
// row repeats a column (`dups`), the cell's ratings share one record: K1's code bits give each array
// exactly one live writer per cell (the reference's dense arrays are last-write-wins), so the record
// ORs the codes of the cell's entries and takes the value from the CODE_IN writer and the entry index
// (-> dy) from the CODE_TGT writer; the list is zeroed first, so a field without a writer reads 0.
// Three small kernels beside K2 / K3 on a low-priority stream, or ahead of the step on the batch's.
//
// K4b (k_row_update) one warp per task, persistent grid: issue the loads of the weight row and its
//              optimizer state, accumulate the gradient from the matched activations
//                decoder:  g = sum_b dy[b,c] * h[b,:]        encoder:  g = sum_b x0[b,blk*N+c] * dz[b,:]
//              in registers, apply the update, store. W and state are read once and written once
//              (16 B/param for Adagrad/RMSprop, 24 for Adam), only for rows that change.
// ============================================================================================
struct SortArgs {
  BatchDev bt;
  int* cnt; int* codeor;                    // [n_cols] each, zeroed per step
  int2* colinfo;                            // [n_cols] (first match, matches) of a touched column
  uint32_t* bits; int W;                    // presence bitmap [n_cols][W words], zeroed per step
  int* counters;                            // [0] matches [1] tasks [2] heavy tasks
  uint32_t* matches; int4* tasks; int2* colseg;
  int4* heavy;                              // (column, array, first match, matches) of every task with more than HEAVY_N matches (null: none recorded)
  int n_cols; int nblk; int3 bits3; int dense; int do_dec; int do_enc;
  int dups;                                 // some row of the store repeats a column: one match per (column, batch row), list zeroed
};

__global__ void __launch_bounds__(128) k_sort_count(SortArgs a) {
  const int4 it = a.bt.items[blockIdx.x];
  if ((int)blockIdx.x >= a.bt.hdr->n_items) return;
  const int b = it.x, p0 = it.w;
  for (int i = threadIdx.x; i < it.z; i += 128) {
    const int code = a.bt.codes[p0 + i];
    if (code == 0) continue;
    const int c = a.bt.ent_col[p0 + i];
    if (a.dups) {
      // the first of the row's ratings of this column to set its bit counts the row
      const uint32_t bit = 1u << (b & 31);
      if ((atomicOr(&a.bits[(size_t)c * a.W + (b >> 5)], bit) & bit) == 0u) atomicAdd(&a.cnt[c], 1);
      atomicOr(&a.codeor[c], code);
    } else {
      atomicAdd(&a.cnt[c], 1);
      atomicOr(&a.codeor[c], code);
      atomicOr(&a.bits[(size_t)c * a.W + (b >> 5)], 1u << (b & 31));
    }
  }
}

// A column matched by more than HEAVY_N batch rows is a "heavy" task: one warp walking its matches is a chain of that
// many dependent L2 round trips and becomes the tail of the whole update kernel (popular items of a user-row batch are
// matched by half of its 128 rows). Heavy tasks are listed separately and each is walked by a whole CTA.
constexpr int HEAVY_N = 24;

__global__ void __launch_bounds__(256) k_sort_alloc(SortArgs a) {
  pdl_trigger();
  pdl_wait();
  const int c = blockIdx.x * 256 + threadIdx.x;
  const int lane = threadIdx.x & 31;
  int n = 0, n_tasks = 0, n_arr = 0;
  int arr[4];
  if (c < a.n_cols) {
    n = a.cnt[c];
    if (n > 0) {
      // dense updates touch every array of every column, including an input block no rating feeds (the "zeros" aux
      // block, bit 0): k_row_update's dense walk leaves all arrays of a heavy column to the heavy list
      const int any = a.dense ? 0xff : a.codeor[c];
      if (a.do_dec && (any & CODE_TGT)) arr[n_arr++] = 0;
      if (a.do_enc)
        for (int blk = 0; blk < a.nblk; ++blk) {
          const int bit = blk == 0 ? a.bits3.x : (blk == 1 ? a.bits3.y : a.bits3.z);
          if (a.dense || (any & bit)) arr[n_arr++] = 1 + blk;
        }
      if (!a.dense) n_tasks = n_arr;
    }
  }
  if (__ballot_sync(FULL, n > 0) == 0u) return;
  // decoder tasks (array 0, always first in arr[]) fill the task array from the front, encoder tasks from the back:
  // K4b then walks the decoder rows first, while the rows K3 has just read are still in L2
  const int n_front = (n_tasks > 0 && arr[0] == 0) ? 1 : 0;
  const int n_back = n_tasks - n_front;
  int sn = n, stk = n_front, ste = n_back;   // inclusive prefixes over the lanes
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t0 = __shfl_up_sync(FULL, sn, o), t1 = __shfl_up_sync(FULL, stk, o), t2 = __shfl_up_sync(FULL, ste, o);
    if (lane >= o) { sn += t0; stk += t1; ste += t2; }
  }
  int b0 = 0, b1 = 0, b2 = 0;
  if (lane == 31) {
    b0 = atomicAdd(&a.counters[0], sn);
    if (stk) b1 = atomicAdd(&a.counters[1], stk);
    if (ste) b2 = atomicAdd(&a.counters[5], ste);
  }
  b0 = __shfl_sync(FULL, b0, 31); b1 = __shfl_sync(FULL, b1, 31); b2 = __shfl_sync(FULL, b2, 31);
  if (n > 0) {
    const int base = b0 + sn - n, front = b1 + stk - n_front, back = b2 + ste - n_back;
    const int cap = a.n_cols * (a.nblk + 1);
    a.colinfo[c] = make_int2(base, n);
    if (a.dense) a.colseg[c] = make_int2(base, n);
    for (int k = 0; k < n_front; ++k) a.tasks[front + k] = make_int4(c, arr[k], base, n);
    for (int k = 0; k < n_back; ++k) a.tasks[cap - 1 - (back + k)] = make_int4(c, arr[n_front + k], base, n);
    if (n > HEAVY_N && a.heavy != nullptr && n_arr > 0) {
      const int h0 = atomicAdd(&a.counters[2], n_arr);
      for (int k = 0; k < n_arr; ++k) a.heavy[h0 + k] = make_int4(c, arr[k], base, n);
    }
  }
}

__global__ void __launch_bounds__(128) k_sort_place(SortArgs a) {
  pdl_trigger();
  pdl_wait();
  const int4 it = a.bt.items[blockIdx.x];
  if ((int)blockIdx.x >= a.bt.hdr->n_items) return;
  const int b = it.x, p0 = it.w;
  for (int i = threadIdx.x; i < it.z; i += 128) {
    const int p = p0 + i;
    const uint32_t code = a.bt.codes[p];
    if (code == 0) continue;
    const int c = a.bt.ent_col[p];
    const int2 info = a.colinfo[c];
    const uint32_t* bw = a.bits + (size_t)c * a.W;
    int rank = __popc(bw[b >> 5] & ((1u << (b & 31)) - 1u));
    for (int w = 0; w < (b >> 5); ++w) rank += __popc(bw[w]);
    const size_t idx = (size_t)(info.x + rank);
    if (a.dups) {
      // the row's ratings of this column share the record; each field has at most one writer
      atomicOr(&a.matches[idx * 3], (uint32_t)b | (code << 16));
      if (code & CODE_IN) a.matches[idx * 3 + 1] = __float_as_uint(a.bt.ent_val[p]);
      if (code & CODE_TGT) a.matches[idx * 3 + 2] = (uint32_t)p;
    } else {
      a.matches[idx * 3] = (uint32_t)b | (code << 16);
      a.matches[idx * 3 + 1] = __float_as_uint(a.bt.ent_val[p]);
      a.matches[idx * 3 + 2] = (uint32_t)p;
    }
  }
}

struct RowArgs {
  const uint32_t* matches; const int4* tasks; const int2* colseg; const int* counters;
  const float* hdec; const float* dz0; const float* dy;
  float* WdecT; float* Wd_s1; float* Wd_s2;
  float* bdec; float* bd_s1; float* bd_s2;
  float* Wenc; float* We_s1; float* We_s2;
  float* Gdec; float* Genc; float* gbdec;   // KIND_GRAD: gradient rows instead of updates (row-parallel mode)
  int n_cols; int3 bits; const BatchHdr* bt_hdr;
  int dense; int n_arr; int arr_map[4];
  const int4* heavy;                        // tasks with more than HEAVY_N matches, walked by whole CTAs (null: every task is a warp's)
  int task_cap;                             // capacity of the task array: task t >= counters[1] is tasks[task_cap - 1 - (t - counters[1])] (K4a puts the encoder tasks there)
  int only;                                 // task list shared by two launches (decoder and encoder rows of different widths): 1 = decoder tasks only, 2 = encoder tasks only
  OptDev opt;
};

constexpr int KIND_GRAD = 4;              // k_row_update: store the gradient row, apply nothing

// WIDE: two matched activation rows in flight per step of a task's walk (more registers, fewer resident warps): for
// catalogues whose weights sit in L2, where the kernel is bound by the longest column's chain of dependent L2 round
// trips instead of by HBM.
// HEAVY: the CTA-cooperative walk of heavy tasks is compiled in (catalogues whose weights are within reach of L2, where
// the longest chain is the kernel's tail; the HBM-bound catalogues keep the lean kernel: no shared memory, 80 registers).
template <int NV, int KIND, bool WIDE, bool HEAVY>
__global__ void __launch_bounds__(256, WIDE ? (NV <= 4 ? 2 : 1) : (KIND == OCF_OPT_ADAM ? (NV <= 4 ? 2 : 1) : (NV <= 4 ? 3 : 2)))
k_row_update(RowArgs a) {
  pdl_trigger();
  pdl_wait();
  constexpr int HP = NV * 128;
  constexpr bool LOAD_W = KIND != KIND_GRAD;
  // Lean variant (catalogues far beyond L2): optimizer state is read once and every row is written once per step, so
  // both go through L2 as evict-first traffic (ld/st.global.cs). What then stays in L2 across kernels are the weight
  // rows K3 has just read: the decoder tasks come first in the list (k_sort_alloc) and find them there.
  constexpr bool STREAM = !WIDE && !HEAVY && KIND != KIND_GRAD;
  __shared__ float4 hpart[HEAVY ? 8 : 1][HEAVY ? HP / 4 : 1];       // heavy tasks: the eight warps' partial gradient rows
  __shared__ float hcs[8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

  // where a task's row lives
  auto row_of = [&](int c, int arr) -> size_t { return arr == 0 ? (size_t)c * HP : ((size_t)(arr - 1) * a.n_cols + c) * HP; };
  // the row and its state: these are the HBM loads, issued before the match walk so that it overlaps them
  auto load_row = [&](int arr, size_t r, float4 (&w)[NV], float4 (&t1)[NV], float4 (&t2)[NV]) {
    const float* Wrow = (arr == 0 ? a.WdecT : a.Wenc) + r + lane * 4;
    const float* S1row = (arr == 0 ? a.Wd_s1 : a.We_s1);
    const float* S2row = (arr == 0 ? a.Wd_s2 : a.We_s2);
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      w[v] = LOAD_W ? *reinterpret_cast<const float4*>(Wrow + v * 128) : make_float4(0.f, 0.f, 0.f, 0.f);
      if (STREAM) {
        t1[v] = KIND != OCF_OPT_SGD ? __ldcs(reinterpret_cast<const float4*>(S1row + r + lane * 4 + v * 128)) : make_float4(0.f, 0.f, 0.f, 0.f);
        t2[v] = KIND == OCF_OPT_ADAM ? __ldcs(reinterpret_cast<const float4*>(S2row + r + lane * 4 + v * 128)) : make_float4(0.f, 0.f, 0.f, 0.f);
      } else {
        t1[v] = (LOAD_W && KIND != OCF_OPT_SGD) ? *reinterpret_cast<const float4*>(S1row + r + lane * 4 + v * 128) : make_float4(0.f, 0.f, 0.f, 0.f);
        t2[v] = KIND == OCF_OPT_ADAM ? *reinterpret_cast<const float4*>(S2row + r + lane * 4 + v * 128) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
  };
  // g += sum over matches [i_begin, i_end) of the task of coef * X[b, :], in match order
  auto walk = [&](int arr, int base, int i_begin, int i_end, float4 (&g)[NV], float& cs) {
    const float* X = (arr == 0 ? a.hdec : a.dz0) + lane * 4;
    const uint32_t bit = arr == 0 ? CODE_TGT : (arr == 1 ? a.bits.x : (arr == 2 ? a.bits.y : a.bits.z));
    for (int i0 = i_begin; i0 < i_end; i0 += 32) {
      // lanes fetch up to 32 match records, then the warp walks them in order
      uint32_t bc = 0; float coef = 0.f;
      if (i0 + lane < i_end) {
        const uint32_t* rec = a.matches + (size_t)(base + i0 + lane) * 3;
        bc = rec[0];
        coef = arr == 0 ? __ldg(a.dy + rec[2]) : (arr == 1 ? __uint_as_float(rec[1]) : __ldg(&a.bt_hdr->aux_value));
      }
      unsigned m = __ballot_sync(FULL, ((bc >> 16) & bit) != 0);
      while (!WIDE && m) {
        const int j = __ffs(m) - 1; m &= m - 1;
        const uint32_t b = __shfl_sync(FULL, bc, j) & 0xffffu;
        const float cf = __shfl_sync(FULL, coef, j);
        const float* x = X + (size_t)b * HP;
#pragma unroll
        for (int v = 0; v < NV; ++v) fma4(g[v], cf, ldg4(x + v * 128));
        cs += cf;
      }
      while (WIDE && m) {
        // two matched rows in flight; the sums keep their order: match j0 is added before match j1
        const int j0 = __ffs(m) - 1; m &= m - 1;
        const bool two = m != 0;
        const int j1 = two ? __ffs(m) - 1 : j0; m &= m - 1;
        const uint32_t b0 = __shfl_sync(FULL, bc, j0) & 0xffffu, b1 = __shfl_sync(FULL, bc, j1) & 0xffffu;
        const float cf0 = __shfl_sync(FULL, coef, j0);
        const float cf1 = two ? __shfl_sync(FULL, coef, j1) : 0.f;
        const float* x0 = X + (size_t)b0 * HP;
        const float* x1 = X + (size_t)b1 * HP;
        float4 a0[NV], a1[NV];
#pragma unroll
        for (int v = 0; v < NV; ++v) { a0[v] = ldg4(x0 + v * 128); a1[v] = ldg4(x1 + v * 128); }
#pragma unroll
        for (int v = 0; v < NV; ++v) { fma4(g[v], cf0, a0[v]); fma4(g[v], cf1, a1[v]); }
        cs += cf0; cs += cf1;
      }
    }
  };
  // gradient row g (and the column's dy sum cs) -> stored (KIND_GRAD) or applied through the optimizer
  auto finish = [&](int c, int arr, size_t r, float4 (&g)[NV], float cs, float4 (&w)[NV], float4 (&t1)[NV], float4 (&t2)[NV]) {
    if (KIND == KIND_GRAD) {
      float* Grow = (arr == 0 ? a.Gdec : a.Genc) + r + lane * 4;
#pragma unroll
      for (int v = 0; v < NV; ++v) *reinterpret_cast<float4*>(Grow + v * 128) = g[v];
      if (arr == 0 && lane == 0) a.gbdec[c] = cs;
      return;
    }
    float* Wrow = (arr == 0 ? a.WdecT : a.Wenc) + r + lane * 4;
    float* S1row = (arr == 0 ? a.Wd_s1 : a.We_s1);
    float* S2row = (arr == 0 ? a.Wd_s2 : a.We_s2);
    const float lr = __ldg(&a.opt.st->lr);      // this step's learning rate (device-resident: a replayed graph carries no scalars)
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      opt_apply_k<KIND>(a.opt, lr, g[v].x, w[v].x, t1[v].x, t2[v].x);
      opt_apply_k<KIND>(a.opt, lr, g[v].y, w[v].y, t1[v].y, t2[v].y);
      opt_apply_k<KIND>(a.opt, lr, g[v].z, w[v].z, t1[v].z, t2[v].z);
      opt_apply_k<KIND>(a.opt, lr, g[v].w, w[v].w, t1[v].w, t2[v].w);
      if (STREAM) {
        __stcs(reinterpret_cast<float4*>(Wrow + v * 128), w[v]);
        if (KIND != OCF_OPT_SGD) __stcs(reinterpret_cast<float4*>(S1row + r + lane * 4 + v * 128), t1[v]);
        if (KIND == OCF_OPT_ADAM) __stcs(reinterpret_cast<float4*>(S2row + r + lane * 4 + v * 128), t2[v]);
      } else {
        *reinterpret_cast<float4*>(Wrow + v * 128) = w[v];
        if (KIND != OCF_OPT_SGD) *reinterpret_cast<float4*>(S1row + r + lane * 4 + v * 128) = t1[v];
        if (KIND == OCF_OPT_ADAM) *reinterpret_cast<float4*>(S2row + r + lane * 4 + v * 128) = t2[v];
      }
    }
    if (arr == 0 && lane == 0) {          // decoder bias: column-local gradient sum_b dy[b,c]
      OptDev ob = a.opt; ob.l2x2 = 0.f;   // Keras regularises kernels only
      float wb = a.bdec[c], b1 = KIND != OCF_OPT_SGD ? a.bd_s1[c] : 0.f, b2 = KIND == OCF_OPT_ADAM ? a.bd_s2[c] : 0.f;
      opt_apply_k<KIND>(ob, lr, cs, wb, b1, b2);
      a.bdec[c] = wb;
      if (KIND != OCF_OPT_SGD) a.bd_s1[c] = b1;
      if (KIND == OCF_OPT_ADAM) a.bd_s2[c] = b2;
    }
  };

  // ---- heavy tasks first (they are the long poles): one CTA each, its eight warps split the match list -------
  const int n_heavy = (HEAVY && a.heavy != nullptr) ? a.counters[2] : 0;
  for (int h = blockIdx.x; HEAVY && h < n_heavy; h += gridDim.x) {
    const int4 task = a.heavy[h];
    const int c = task.x, arr = task.y, base = task.z, n = task.w;
    if (a.only != 0 && (a.only == 1) != (arr == 0)) continue;            // CTA-uniform
    const size_t r = row_of(c, arr);
    float4 w[NV], t1[NV], t2[NV], g[NV];
    if (warp == 0) load_row(arr, r, w, t1, t2);
#pragma unroll
    for (int v = 0; v < NV; ++v) g[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    float cs = 0.f;
    const int per = (n + 7) >> 3;
    walk(arr, base, min(n, warp * per), min(n, (warp + 1) * per), g, cs);
#pragma unroll
    for (int v = 0; v < NV; ++v) hpart[warp][v * 32 + lane] = g[v];
    if (lane == 0) hcs[warp] = cs;
    __syncthreads();
    if (warp == 0) {
      cs = hcs[0];
#pragma unroll
      for (int v = 0; v < NV; ++v) g[v] = hpart[0][v * 32 + lane];
      for (int k = 1; k < 8; ++k) {                                    // warp order = match order of the eight segments
        cs += hcs[k];
#pragma unroll
        for (int v = 0; v < NV; ++v) {
          const float4 p = hpart[k][v * 32 + lane];
          g[v].x += p.x; g[v].y += p.y; g[v].z += p.z; g[v].w += p.w;
        }
      }
      finish(c, arr, r, g, cs, w, t1, t2);
    }
    __syncthreads();
  }

  // ---- every other task: one warp each ------------------------------------------------------------------------
  const int n_front = a.dense ? 0 : a.counters[1];
  const long long n_tasks = a.dense ? (long long)a.n_cols * a.n_arr : (long long)n_front + a.counters[5];
  auto task_at = [&](long long t) -> int4 { return a.tasks[t < n_front ? t : (long long)a.task_cap - 1 - (t - n_front)]; };
  auto run_task = [&](int c, int arr, int base, int n) {
    const size_t r = row_of(c, arr);
    float4 w[NV], t1[NV], t2[NV], g[NV];
    load_row(arr, r, w, t1, t2);
#pragma unroll
    for (int v = 0; v < NV; ++v) g[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    float cs = 0.f;
    walk(arr, base, 0, n, g, cs);
    finish(c, arr, r, g, cs, w, t1, t2);
  };
  if constexpr (!WIDE && !HEAVY && KIND != KIND_GRAD) {
    // Lean variant (catalogues far beyond L2, hundreds of tasks per warp): tasks are dealt out in chunks of 4 through
    // a cursor (zeroed with the work list's counters), so a warp that drew long match lists simply takes fewer
    // chunks and the kernel has no tail of unlucky warps (Netflix shape: 1.75 -> 1.56 ms, 0.81 -> 0.91 of HBM).
    // The cursor for the next chunk is bumped before the current chunk is processed (its round trip hides behind
    // the chunk), and the chunk's four task descriptors arrive in one load.
    int* cursor = const_cast<int*>(a.counters) + (a.only == 2 ? 4 : 3);
    int pend = lane == 0 ? atomicAdd(cursor, 4) : 0;
    for (;;) {
      const long long t0 = __shfl_sync(FULL, pend, 0);
      if (t0 >= n_tasks) break;
      if (lane == 0) pend = atomicAdd(cursor, 4);
      int4 mine = make_int4(0, 0, 0, 0);
      if (lane < 4 && t0 + lane < n_tasks) {
        if (a.dense) {
          const long long t = t0 + lane;
          const int c = (int)(t / a.n_arr);
          const int2 seg = a.colseg[c];
          mine = make_int4(c, a.arr_map[t - (long long)c * a.n_arr], seg.x, seg.y);
        } else {
          mine = task_at(t0 + lane);
        }
      }
      const int cnt = (int)min((long long)4, n_tasks - t0);
      for (int k = 0; k < cnt; ++k) {
        const int c = __shfl_sync(FULL, mine.x, k), arr = __shfl_sync(FULL, mine.y, k);
        const int base = __shfl_sync(FULL, mine.z, k), n = __shfl_sync(FULL, mine.w, k);
        if (!a.dense && a.only != 0 && (a.only == 1) != (arr == 0)) continue;
        run_task(c, arr, base, n);
      }
    }
  } else {
    const int gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    for (long long t = gwarp; t < n_tasks; t += nwarps) {
      int c, arr, base, n;
      if (a.dense) {
        c = (int)(t / a.n_arr); arr = a.arr_map[t - (long long)c * a.n_arr];
        const int2 seg = a.colseg[c]; base = seg.x; n = seg.y;
      } else {
        const int4 task = task_at(t);
        c = task.x; arr = task.y; base = task.z; n = task.w;
        if (a.only != 0 && (a.only == 1) != (arr == 0)) continue;
      }
      if (HEAVY && a.heavy != nullptr && n > HEAVY_N) continue;            // done above by a whole CTA
      run_task(c, arr, base, n);
    }
  }
}

// Row-parallel (data-parallel) mode: the gradients of all ranks are summed by an all-reduce
// first, so the optimizer runs as a plain stream over (parameter, gradient, state): 20 B/param
// for Adagrad/RMSprop, 28 for Adam. n is a multiple of 4 for kernels; biases take the scalar tail.
__global__ void __launch_bounds__(256)
k_dense_update(float* __restrict__ w, const float* __restrict__ g, float* __restrict__ s1, float* __restrict__ s2,
               size_t n, OptDev o) {
  const float lr = o.st->lr;
  const size_t n4 = n / 4;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 wv = reinterpret_cast<float4*>(w)[i];
    const float4 gv = reinterpret_cast<const float4*>(g)[i];
    float4 a = s1 ? reinterpret_cast<float4*>(s1)[i] : make_float4(0.f, 0.f, 0.f, 0.f);
    float4 b = s2 ? reinterpret_cast<float4*>(s2)[i] : make_float4(0.f, 0.f, 0.f, 0.f);
    opt_apply(o, lr, gv.x, wv.x, a.x, b.x); opt_apply(o, lr, gv.y, wv.y, a.y, b.y);
    opt_apply(o, lr, gv.z, wv.z, a.z, b.z); opt_apply(o, lr, gv.w, wv.w, a.w, b.w);
    reinterpret_cast<float4*>(w)[i] = wv;
    if (s1) reinterpret_cast<float4*>(s1)[i] = a;
    if (s2) reinterpret_cast<float4*>(s2)[i] = b;
  }
  for (size_t i = n4 * 4 + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    float wv = w[i], a = s1 ? s1[i] : 0.f, b = s2 ? s2[i] : 0.f;
    opt_apply(o, lr, g[i], wv, a, b);
    w[i] = wv;
    if (s1) s1[i] = a;
    if (s2) s2[i] = b;
  }
}

// Sum of squares of a kernel (for the L2 term of the reported loss), 64 fixed partials.
__global__ void __launch_bounds__(256) k_sumsq(const float* __restrict__ w, size_t n, float* __restrict__ part) {
  __shared__ float sh[8];
  float s = 0.f;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    s = fmaf(w[i], w[i], s);
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int k = 0; k < 8; ++k) t += sh[k];
    part[blockIdx.x] = t;
  }
}

// Per-step metric record from the per-row statistics (train.py:102-121 + the Keras loss).
// One warp, fixed summation order.
__device__ void metrics_record(const MetricArgs& a, int lane) {
  float sse = 0.f, sae = 0.f, cnt = 0.f, srt = 0.f, reg = 0.f;
  for (int b = lane; b < a.rows; b += 32) {
    const float s = a.rowstats[b * ROWSTAT_W];
    sse += s; sae += a.rowstats[b * ROWSTAT_W + 1]; cnt += a.rowstats[b * ROWSTAT_W + 2];
    srt += sqrtf(s);
  }
  for (int k = lane; k < a.n_reg; k += 32) reg += a.regparts[k];
  sse = warp_sum(sse); sae = warp_sum(sae); cnt = warp_sum(cnt); srt = warp_sum(srt); reg = warp_sum(reg);
  if (lane == 0) {
    const int slot = a.st->log_slot;
    float* rec = a.log + (size_t)slot * LOG_W;
    const float bn = a.rows_total * a.n_cols_total;
    const float mse = sse / bn, mae = sae / bn;
    const float acc_mae = sae / cnt;
    rec[0] = (a.loss_kind == OCF_LOSS_MSE ? mse : mae) + (a.n_reg > 0 ? a.l2 * reg : 0.f);
    rec[1] = mae;
    rec[2] = acc_mae;
    rec[3] = acc_mae / a.rating_range;
    rec[4] = sqrtf(a.rows_total / cnt) * srt / a.rows_total;
    rec[5] = sse / cnt;
    rec[6] = sse;
    rec[7] = cnt;
    __threadfence_system();
    a.st->log_slot = slot + 1 == LOG_CAP ? 0 : slot + 1;
    if (a.advance_step) a.st->step += 1u;
  }
}

// Rewrites the model's device-resident step scalars (only when a caller's step arguments differ
// from what the device would use next).
__global__ void k_set_step(StepDev* st, StepDev v) { *st = v; }

__global__ void __launch_bounds__(32) k_metrics(MetricArgs a) { metrics_record(a, threadIdx.x); }

}  // namespace ocf
