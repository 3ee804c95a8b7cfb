// Shared definitions of libocf_b200: error handling, device-side structs, small device helpers.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <string>

#include "../../include/ocf.h"

namespace ocf {

// ---- error plumbing ---------------------------------------------------------------------
std::string& last_error();
int fail(int code, const std::string& msg);

#define OCF_CUDA(expr)                                                                   \
  do {                                                                                   \
    cudaError_t _e = (expr);                                                             \
    if (_e != cudaSuccess)                                                               \
      return ::ocf::fail(OCF_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); \
  } while (0)

#define OCF_REQUIRE(cond, msg)                                      \
  do {                                                              \
    if (!(cond)) return ::ocf::fail(OCF_ERR_INVALID, (msg));        \
  } while (0)

#define OCF_TRY(expr)            \
  do {                           \
    int _s = (expr);             \
    if (_s != OCF_OK) return _s; \
  } while (0)

extern std::atomic<long long> g_launches;
#define OCF_LAUNCHED()                                                                       \
  do {                                                                                       \
    ::ocf::g_launches.fetch_add(1, std::memory_order_relaxed);                               \
    cudaError_t _e = cudaGetLastError();                                                     \
    if (_e != cudaSuccess)                                                                   \
      return ::ocf::fail(OCF_ERR_CUDA, std::string("kernel launch: ") + cudaGetErrorString(_e)); \
  } while (0)

// ---- per-entry code bits written by the gather kernels (K1) --------------------------------
// An entry is "live" for an array when it is the last rating of its row that writes that array
// at that column (the dense fills in data_reader.py:158-169 are last-write-wins).
constexpr uint8_t CODE_IN = 1;    // contributes ratings_batch_inputs / mask_batch_inputs
constexpr uint8_t CODE_OBS = 2;   // contributes missing_data_mask
constexpr uint8_t CODE_TGT = 4;   // contributes ratings_batch_targets / mask_batch_targets

constexpr int MAX_BATCH_ROWS = 4096;
constexpr int HPAD = 128;                 // hidden widths are padded to a multiple of 128 floats
constexpr int MAX_HP = 1024;
constexpr int ROWSTAT_W = 4;              // sse, sae, cnt, unused

// Device view of a rating store.
struct StoreDev {
  const int64_t* rowptr;
  const int32_t* col;
  const float* val;
  const int32_t* next_dup;   // index inside the row of the next later rating of the same column, or -1; null if no row repeats a column
  const int32_t* orig_pos;   // column shards: position of the entry inside its FULL row (null: the store holds full rows)
};

// What changes from one fill of a batch object to the next, as the device sees it: the first bytes of
// the batch's staging buffer, uploaded with the row ids. Kernels of a captured step (CUDA graph) read
// their sizes here, so a replayed graph needs no per-step parameter update; every pointer in BatchDev
// is fixed for the life of the batch object.
struct BatchHdr {
  int B;
  int n_items;
  int n_entries;
  uint32_t pad0;
  int cdf_row0;              // device-RNG mode: index of batch row 0 among the drawing unit's sparsity draws
  int pass_through;
  double rng_lo, rng_range;  // np.random.uniform(lo, hi) of the rows' sparsity draws (range = hi - lo)
  float aux_value;
  uint32_t word_base;        // device-RNG mode: ring position of the batch's first stream word
  uint32_t ring_words;       //   size of the stream ring in words
  int pad[3];
};
static_assert(sizeof(BatchHdr) == 64, "BatchHdr is one 64-byte block at the head of the staging buffer");

// Per-step scalars of a model, resident in device memory so that a captured step replays unchanged:
// the dropout counter, the slot of the metric log the step writes, the step's learning rate (decay /
// Adam bias correction folded in). The step's last kernel advances step and log_slot; the host keeps a
// mirror and rewrites the struct (k_set_step) only when a caller's arguments differ from it.
struct StepDev {
  uint32_t step;
  int32_t log_slot;
  float lr;
  uint32_t seed_lo, seed_hi;
  int32_t pad[3];
};

// Device view of one batch. The first group is uploaded by the host in one copy, the second
// is written by K1. B / n_items / n_entries are the host's copy of the current fill (for host logic
// and for kernels launched outside captured steps); captured kernels use hdr.
struct BatchDev {
  const BatchHdr* hdr;
  int B;
  int n_items;
  int n_entries;
  const int32_t* row_ids;    // [B] store row of batch row b
  const int32_t* ent_off;    // [B+1] first entry of batch row b
  const int32_t* in_len;     // [B] fixed-split: how many of the row's entries come from the input store
  const int4* items;         // [n_items] (b, start, len, first entry = ent_off[b] + start): a chunk of a row's entries
  const int32_t* item_ptr;   // [B+1] items of row b
  const uint8_t* flags;      // [n_entries] keep flags (split mode)
  const int32_t* draw_off;   // [B] device-RNG mode: index of the row's first draw in the batch's slice of the stream
  const uint32_t* words;     //     the generator's stream ring (tempered MT19937 words; 2 per draw)
  double rng_lo, rng_range;  //     np.random.uniform(lo, hi) of the rows' sparsity draws (range = hi - lo)
  int cdf_row0;              //     index of batch row 0 among the drawing unit's sparsity draws
  uint8_t* flags_out;        // [n_entries] == flags; written by K1 in device-RNG mode
  int32_t* ent_col;          // [n_entries]
  float* ent_val;            // [n_entries]
  uint8_t* codes;            // [n_entries]
};

struct OptDev {
  int kind;          // ocf_optimizer
  float lr;          // host's copy of this step's learning rate; kernels use st->lr (passed to opt_apply as `lr`)
  float p1;          // rho / beta_1
  float one_m_p1;    // 1 - rho / 1 - beta_1 (computed in double on the host, like Keras)
  float p2;          // beta_2
  float one_m_p2;
  float eps;
  float l2x2;        // 2 * lambda, 0 without regularisation
  int dense;         // 1: every parameter changes every step (RMSprop, Adam, L2)
  const StepDev* st; // kernels take this step's lr from st->lr (the value above is the host's copy)
};

// sqrt / divide of the update rules use the MUFU approximations (<= 2 ulp): the IEEE-rounded
// versions cost ~5x the instructions and made the update kernel issue-bound (profiles/r01).
__device__ __forceinline__ float fast_sqrt(float x) {
  float r;
  asm("sqrt.approx.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

template <int KIND>
__device__ __forceinline__ void opt_apply_k(const OptDev& o, const float lr, float g, float& w, float& s1, float& s2) {
  g = fmaf(o.l2x2, w, g);
  if (KIND == OCF_OPT_SGD) {
    w = fmaf(-lr, g, w);
  } else if (KIND == OCF_OPT_ADAGRAD) {
    s1 = fmaf(g, g, s1);
    w -= __fdividef(lr * g, fast_sqrt(s1) + o.eps);
  } else if (KIND == OCF_OPT_RMSPROP) {
    s1 = fmaf(o.one_m_p1 * g, g, o.p1 * s1);
    w -= __fdividef(lr * g, fast_sqrt(s1) + o.eps);
  } else {  // Adam
    s1 = fmaf(o.one_m_p1, g, o.p1 * s1);
    s2 = fmaf(o.one_m_p2 * g, g, o.p2 * s2);
    w -= __fdividef(lr * s1, fast_sqrt(s2) + o.eps);
  }
}

__device__ __forceinline__ void opt_apply(const OptDev& o, const float lr, float g, float& w, float& s1, float& s2) {
  switch (o.kind) {
    case OCF_OPT_SGD: opt_apply_k<OCF_OPT_SGD>(o, lr, g, w, s1, s2); break;
    case OCF_OPT_ADAGRAD: opt_apply_k<OCF_OPT_ADAGRAD>(o, lr, g, w, s1, s2); break;
    case OCF_OPT_RMSPROP: opt_apply_k<OCF_OPT_RMSPROP>(o, lr, g, w, s1, s2); break;
    default: opt_apply_k<OCF_OPT_ADAM>(o, lr, g, w, s1, s2); break;
  }
}

__device__ __forceinline__ float act_fwd(int kind, float z) {
  switch (kind) {
    case OCF_ACT_SIGMOID: return 1.0f / (1.0f + expf(-z));
    case OCF_ACT_TANH: return tanhf(z);
    case OCF_ACT_RELU: return fmaxf(z, 0.0f);
    case OCF_ACT_ELU: return z > 0.0f ? z : expm1f(z);
    case OCF_ACT_SELU: return 1.0507009873554805f * (z > 0.0f ? z : 1.6732632423543772f * expm1f(z));
    case OCF_ACT_SOFTPLUS: return fmaxf(z, 0.0f) + log1pf(expf(-fabsf(z)));
    default: return z;
  }
}

// d act / d z expressed through the activation value a (all supported activations allow it).
__device__ __forceinline__ float act_bwd(int kind, float a) {
  switch (kind) {
    case OCF_ACT_SIGMOID: return a * (1.0f - a);
    case OCF_ACT_TANH: return 1.0f - a * a;
    case OCF_ACT_RELU: return a > 0.0f ? 1.0f : 0.0f;
    case OCF_ACT_ELU: return a > 0.0f ? 1.0f : a + 1.0f;
    case OCF_ACT_SELU: return a > 0.0f ? 1.0507009873554805f : a + 1.0507009873554805f * 1.6732632423543772f;
    case OCF_ACT_SOFTPLUS: return 1.0f - expf(-a);
    default: return 1.0f;
  }
}

// Philox4x32-10; the dropout-mask specification is in oracle/philox.py.
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}

// NumPy's next_double for MT19937: 53 bits from two consecutive tempered words.
__device__ __forceinline__ double mt_double(uint32_t a, uint32_t b) {
  return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6)) * (1.0 / 9007199254740992.0);
}

// Programmatic dependent launch (PDL). A kernel launched with the programmatic-stream-serialization attribute may
// become resident while its predecessor in the stream still runs: `pdl_trigger` (first statement) lets the NEXT
// kernel do so as soon as every CTA of this grid has started, `pdl_wait` blocks until the PREVIOUS grid has
// completed and its writes are visible - nothing the predecessor produces may be read before it. Between two
// dependent small kernels this hides the launch latency and the prologue (a training step of the small catalogues
// is a chain of 9-13 such kernels). Both are no-ops in a launch without the attribute.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void fma4(float4& a, float s, const float4& w) {
  a.x = fmaf(s, w.x, a.x); a.y = fmaf(s, w.y, a.y); a.z = fmaf(s, w.z, a.z); a.w = fmaf(s, w.w, a.w);
}
__device__ __forceinline__ float dot4(const float4& a, const float4& b, float acc) {
  acc = fmaf(a.x, b.x, acc); acc = fmaf(a.y, b.y, acc); acc = fmaf(a.z, b.z, acc); return fmaf(a.w, b.w, acc);
}

}  // namespace ocf
