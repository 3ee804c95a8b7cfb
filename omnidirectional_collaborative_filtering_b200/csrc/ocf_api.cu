// libocf_b200: the C ABI of include/ocf.h over the kernels in ocf_kernels.cuh.
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <tuple>
#include <vector>

#include "ocf_kernels.cuh"
#include "ocf_mtjump.h"
#include "ocf_score_tc.cuh"
#include "ocf_gemm_tc.cuh"
#include "ocf_topk.cuh"
#include "ocf_rank.cuh"

namespace ocf {

std::string& last_error() {
  static thread_local std::string e;
  return e;
}
int fail(int code, const std::string& msg) {
  last_error() = msg;
  return code;
}
std::atomic<long long> g_launches{0};
static std::atomic<int> g_comms_alive{0};      // NCCL communicators of this process (ocf_comm_create / _destroy)

static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }
static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
static inline int pad_h(int h) { return (int)align_up((size_t)h, HPAD); }

// Device allocations of one handle, freed together.
struct Arena {
  std::vector<void*> ptrs;
  size_t bytes = 0;
  int alloc(void** out, size_t n, bool zero) {
    *out = nullptr;
    if (n == 0) n = 16;
    cudaError_t e = cudaMalloc(out, n);
    if (e != cudaSuccess) return fail(OCF_ERR_NOMEM, std::string("cudaMalloc(") + std::to_string(n) + "): " + cudaGetErrorString(e));
    ptrs.push_back(*out);
    bytes += n;
    if (zero) OCF_CUDA(cudaMemset(*out, 0, n));
    return OCF_OK;
  }
  template <typename T> int get(T** out, size_t count, bool zero = false) {
    return alloc(reinterpret_cast<void**>(out), count * sizeof(T), zero);
  }
  void release() {
    for (void* p : ptrs) cudaFree(p);
    ptrs.clear();
    bytes = 0;
  }
};

// NCCL is loaded at run time (the library must load, and every single-GPU path must work, on a
// box without it): the copy PyTorch already mapped into the process when there is one, else the
// system's libnccl.so.2.
struct NcclApi {
  decltype(&ncclGetUniqueId) getUniqueId = nullptr;
  decltype(&ncclCommInitRank) commInitRank = nullptr;
  decltype(&ncclCommDestroy) commDestroy = nullptr;
  decltype(&ncclAllReduce) allReduce = nullptr;
  decltype(&ncclAllGather) allGather = nullptr;
  decltype(&ncclGetErrorString) getErrorString = nullptr;
  bool ok = false;
};
static NcclApi& nccl_api() {
  static NcclApi api = [] {
    NcclApi a;
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) return a;
    a.getUniqueId = reinterpret_cast<decltype(a.getUniqueId)>(dlsym(h, "ncclGetUniqueId"));
    a.commInitRank = reinterpret_cast<decltype(a.commInitRank)>(dlsym(h, "ncclCommInitRank"));
    a.commDestroy = reinterpret_cast<decltype(a.commDestroy)>(dlsym(h, "ncclCommDestroy"));
    a.allReduce = reinterpret_cast<decltype(a.allReduce)>(dlsym(h, "ncclAllReduce"));
    a.allGather = reinterpret_cast<decltype(a.allGather)>(dlsym(h, "ncclAllGather"));
    a.getErrorString = reinterpret_cast<decltype(a.getErrorString)>(dlsym(h, "ncclGetErrorString"));
    a.ok = a.getUniqueId && a.commInitRank && a.commDestroy && a.allReduce && a.allGather && a.getErrorString;
    return a;
  }();
  return api;
}
#define OCF_NCCL(expr)                                                                        \
  do {                                                                                        \
    ncclResult_t _r = (expr);                                                                 \
    if (_r != ncclSuccess)                                                                    \
      return ::ocf::fail(OCF_ERR_CUDA, std::string(#expr) + ": " + nccl_api().getErrorString(_r)); \
  } while (0)

}  // namespace ocf

using namespace ocf;

struct ocf_comm {
  ncclComm_t comm = nullptr;
  int rank = 0, world = 1, device = 0;
};

// ============================================================================================
// handles
// ============================================================================================
struct ocf_store {
  int64_t n_rows = 0, n_cols = 0, nnz = 0;
  bool has_dups = false;
  std::vector<int64_t> h_rowptr;
  StoreDev dev{};
  Arena mem;
};

// NumPy's MT19937 stream as a service on the device. The stream is addressed by absolute word position u, counted
// from the start of the ORIGIN array (the 624-word key of the last set_state; its words are u = 0..623, the stream
// continues at u = pos). Regeneration g >= 1 of the origin array is words [624 g, 624 g + 624). Blocks of C
// regenerations (block k = regenerations 1 + kC .. (k+1)C) are produced by M worker CTAs: worker k % M makes block k
// on its own CUDA stream and then jumps its array over the other workers' M - 1 blocks (k_mt_jump_apply). All words
// land in one ring of R blocks, addressed (u mod ring words). The host only keeps positions: which blocks are
// enqueued, how far the consumers have read, which event guards which ring slot.
struct ocf_rng {
  int device = 0;
  int M = 1, C = 256, R = 16;                   // workers, regenerations per block, ring blocks
  int64_t BW = 0, RW = 0;                       // words per block / in the ring
  uint32_t* d_ring = nullptr;
  uint32_t* d_arrays = nullptr;                 // [M][2][640] worker arrays (double-buffered by the jumps) + timing words
  uint32_t* d_seq = nullptr;                    // [M][33 * 624] sequence a jump reads
  uint32_t* d_poly = nullptr;                   // [2][624]: x^(624 C) (placement), x^(624 C (M-1)) (steady state)
  std::vector<cudaStream_t> wstream;
  std::vector<cudaEvent_t> block_ev, slot_free;
  std::vector<char> slot_free_valid;
  std::vector<int> cur;                         // which of its two array buffers worker j holds
  cudaEvent_t placed = nullptr;
  cudaStream_t io = nullptr;                    // read-backs of the state: never through the legacy stream, which would wait for every step in flight
  int64_t next_block = 0;                       // first block not enqueued yet
  int64_t pos_u = 0;                            // consumers' position (absolute word)
  uint32_t origin[624] = {0};
  bool have_state = false;
  int last_worker = 0;
  Arena mem;
  uint32_t* array_of(int j, int which) const { return d_arrays + ((size_t)j * 2 + which) * 640; }
};

struct ocf_pair {
  const ocf_store* in = nullptr;
  const ocf_store* tg = nullptr;
  uint8_t* d_in_overlap = nullptr;
  Arena mem;
};

// K4a's product for one batch: what K4b walks. The model owns one (filled inside the step, on a side stream);
// a batch object owns another when its column grouping runs AHEAD of the step on the batch's own stream.
struct WorkList {
  uint32_t* matches = nullptr;    // [3 * entries] (batch row | code << 16, value, entry)
  int64_t entries = 0;            //   capacity of `matches` in records
  int2* seg = nullptr;            // [n_cols] dense mode: (first match, matches) of every column
  int4* tasks = nullptr;          // [(nblk + 1) * n_cols]
  int4* heavy = nullptr;          //   tasks with more than HEAVY_N matches
  int* counters = nullptr;        // [8]: matches, tasks at the front of the task array, heavy tasks, K4b's two task cursors (two launches may share a list), tasks at the back
  int* state = nullptr;           // [2][n_cols] per-column count / code OR
  int2* info = nullptr;           // [n_cols] (first match, matches) of a touched column
  uint32_t* bits = nullptr;       // presence bitmap [n_cols][ceil(rows / 32)]
};

// What a work list depends on besides the batch's own tiles.
struct WorkSig {
  int n_cols = 0, nblk = 0, b0 = 0, b1 = 0, b2 = 0, do_dec = 0, do_enc = 0, dense = 0, heavy = 0, B = 0, dups = 0;
  bool operator==(const WorkSig& o) const {
    return n_cols == o.n_cols && nblk == o.nblk && b0 == o.b0 && b1 == o.b1 && b2 == o.b2 && do_dec == o.do_dec &&
           do_enc == o.do_enc && dense == o.dense && heavy == o.heavy && B == o.B && dups == o.dups;
  }
};

struct ocf_batch {
  uint64_t uid = 0;               // never reused: captured steps are keyed by it
  int max_rows = 0;
  int64_t max_entries = 0;
  int max_items = 0;
  size_t staging_bytes = 0;
  size_t off[8] = {0};            // fixed layout of the staging buffer (staging_layout)
  uint8_t* h_staging = nullptr;   // pinned
  uint8_t* d_staging = nullptr;
  cudaEvent_t copied = nullptr;
  bool copy_pending = false;
  // A fill (staging copy + gather kernel K1) runs on the batch's own stream, so that it overlaps the step the
  // caller's stream is still executing (K1 and its H2D copy were ~10 % of a small catalogue's step). `gathered`
  // orders every consumer after the fill, `consumed` orders the next fill after the last consumer.
  cudaStream_t gstream = nullptr;
  cudaEvent_t gathered = nullptr, consumed = nullptr;
  bool gathered_valid = false, consumed_valid = false;
  int32_t* d_ent_col = nullptr;
  float* d_ent_val = nullptr;
  uint8_t* d_codes = nullptr;
  BatchDev dev{};
  int mode = 0;                   // 0 empty, 1 split, 2 fixed
  const ocf_store* store = nullptr;
  const ocf_pair* pair = nullptr;
  int pass_through = 0;
  float aux_value = -1.f;
  int64_t target_count = 0;
  size_t last_h2d = 0;
  std::vector<uint8_t> flag_scratch;
  // device-RNG mode: where this batch's draws sit in the generator's stream ring, and the per-row cdf
  const uint32_t* d_words = nullptr;   // the ring (owned by the ocf_rng)
  uint32_t word_base = 0, ring_words = 0;
  double rng_lo = 0.0, rng_range = 0.0;
  int64_t draw_base = 0;           // index of the batch's first per-rating draw in its slice of the stream
  int cdf0_row0 = 0;               // row-parallel slice: index of the batch's first row among the sparsity draws
  bool rng_mode = false;
  // The batch's own update work list (K4a): grouped by catalogue column right behind the gather, on the batch's
  // stream, so that it runs under an EARLIER step instead of beside this step's K2 / K3 (which it slowed from 31
  // to 48 us on the ML-10M shape). One zeroed region [counters | state | bits | seg], one memset.
  WorkList wl{};
  Arena wl_mem;
  uint8_t* wl_zero = nullptr;     // start of the zeroed region (= wl.seg)
  int wl_cols = 0, wl_nblk = 0;   // what the allocation was sized for
  WorkSig wl_sig{};               // what the list in `wl` was built for ...
  uint64_t fill_seq = 0, wl_seq = 0;   // ... and for which fill (0: none)
  cudaEvent_t wl_ready = nullptr;
  cudaGraphExec_t wl_graph = nullptr;  // memset + the three K4a kernels of `wl_graph_sig`, one launch
  WorkSig wl_graph_sig{};
  int wl_graph_kernels = 0;
  bool wl_graph_failed = false;
  Arena mem;
};

struct Layer {
  int fan_in = 0, fan_out = 0;    // true sizes (Keras)
  int rows = 0, hp = 0;           // internal: W is [rows, hp] (decoder: [n_cols, hp_in])
  float *W = nullptr, *b = nullptr;
  float *Ws1 = nullptr, *Ws2 = nullptr, *bs1 = nullptr, *bs2 = nullptr;
  int bias_len = 0;
  bool trainable = true;
};

struct ocf_model {
  ocf_model_config cfg{};
  int L = 0, nblk = 1;
  int3 bits{};
  std::vector<Layer> layers;      // 0 = encoder, 1..L-1 hidden, L = decoder
  std::vector<int> hp;            // padded hidden widths
  int max_items = 0;
  // workspaces
  float *P1 = nullptr, *P2 = nullptr, *itemstats = nullptr, *rowstats = nullptr, *dy = nullptr;
  std::vector<float*> zsum, act, h, dscale, dz;
  float* dh_top = nullptr;
  float* dense_out = nullptr;
  float* regparts = nullptr;
  float* h_rec = nullptr;         // page-locked, mapped: the metric log, written by the kernels, read by the host
  float* h_rec_dev = nullptr;     //   its device address
  StepDev* d_step = nullptr;      // device-resident step scalars (dropout counter, log slot, lr)
  StepDev step_mirror{};          //   what the device holds once everything enqueued so far has run
  bool step_mirror_valid = false;
  TailBuf tail{};                 // row-tail counters and group sums of K2 / K3
  // captured steps (CUDA graphs), keyed by batch object / rows / kind / whether the batch's store repeats a
  // column (K4a clears the match list first then); dropped whenever anything they
  // bake in changes (workspaces, optimizer, trainable flags, ...)
  struct StepGraph { cudaGraphExec_t exec = nullptr; int kernels = 0; int seen = 0; bool failed = false; };
  std::map<std::tuple<uint64_t, int, int, int, int, int>, StepGraph> graphs;
  cudaStream_t cap = nullptr;     // capture stream
  bool capturing = false;
  int64_t steps_logged = 0;
  cudaEvent_t step_ev[64] = {nullptr};
  uint32_t* col_matches = nullptr;
  int2* col_seg = nullptr;
  int4* col_tasks = nullptr;
  int4* col_heavy = nullptr;      // tasks with more than HEAVY_N matches, same capacity as col_tasks
  int* col_counters = nullptr;
  int32_t* topk_cols = nullptr;   // top-k epilogue outputs [max_rows, 512] (allocated with dense_out's arena)
  float* topk_scores = nullptr;
  size_t topk_cap = 0;
  // ranking evaluation workspace (ocf_rank.cuh; allocated with dense_out's arena): [max_entries] each
  uint32_t* rank_key = nullptr;
  int32_t *rank_col = nullptr, *rank_ent = nullptr, *rank_cnt = nullptr, *rank_out = nullptr;
  int32_t* rank_nrel = nullptr;   //   [max_rows]
  unsigned long long* rank_ncand = nullptr;
  bool rank_ok = false;
  int* col_state = nullptr;       // batch-side K4a: [2][n_cols] per-column count / code OR, zeroed per step
  int2* col_info = nullptr;       //   [n_cols] (first match, matches)
  uint32_t* col_bits = nullptr;   //   presence bitmap [n_cols][ceil(max_rows / 32)]
  size_t col_bits_words = 0;
  int sm_count = 148;
  // the column scan (K4a) needs only the gathered batch: it runs on a side stream beside K2/K3
  cudaStream_t side = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  bool scan_pending = false;
  // models with hidden layers: the decoder rows' update (needs K3's outputs only) and every hidden layer's gradient
  // product (needs its own dz only) leave the step's critical path on a second side stream
  cudaStream_t side2 = nullptr;
  cudaEvent_t ev_fork2 = nullptr, ev_join2 = nullptr, ev_dz[8] = {nullptr};
  // multi-GPU (ocf_model_set_comm)
  ocf_comm* comm = nullptr;
  int par_mode = 0;               // 0 none, OCF_PAR_COLUMNS, OCF_PAR_ROWS
  float* grads = nullptr;         // row-parallel mode: one arena, per layer [kernel | bias] like the parameters
  size_t grads_count = 0;
  std::vector<float*> gW, gb;
  float* gathered_stats = nullptr;   // [world * max_rows * 4] row statistics of the global batch
  Arena par_mem;
  // tcgen05 scoring: TMA maps of the decoder kernel and of the top activation
  CUtensorMap map_w{}, map_h{};
  bool map_w_ok = false, map_h_ok = false;
  int map_h_box = 0;
  long long act_rows = 0;         // rows the activation buffers hold (max_rows padded to 256)
  // optimizer
  int opt_kind = OCF_OPT_ADAGRAD;
  float lr = 0.005f, p1 = 0.9f, p2 = 0.999f, eps = 1e-8f, decay = 0.f;
  int64_t iterations = 0;
  bool has_s1 = false, has_s2 = false;
  Arena mem, opt_mem, dense_mem, ws_mem;
};

constexpr int N_REGPART = 64;

// Launch with the programmatic-stream-serialization attribute (PDL, ocf_common.cuh): only for kernels that call
// pdl_wait() before they touch memory, and only when the previous operation in the stream is a kernel.
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(bool pdl, void (*kern)(KArgs...), dim3 grid, dim3 block, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = 0; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

static void drop_graphs(ocf_model* m) {
  for (auto& kv : m->graphs)
    if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
  m->graphs.clear();
}

// ============================================================================================
// misc
// ============================================================================================
extern "C" const char* ocf_last_error(void) { return last_error().c_str(); }
extern "C" int ocf_version(void) { return OCF_VERSION; }
extern "C" int ocf_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}
extern "C" int64_t ocf_kernel_launches(void) { return (int64_t)g_launches.load(); }

// Page-locked host memory for buffers that cross PCIe every call (score / predict outputs):
// copies to pageable memory are staged by the driver at a fraction of the link's bandwidth.
extern "C" int ocf_host_alloc(int64_t bytes, void** out) {
  OCF_REQUIRE(out != nullptr && bytes >= 0, "ocf_host_alloc: bad argument");
  *out = nullptr;
  if (cudaMallocHost(out, (size_t)std::max<int64_t>(bytes, 16)) != cudaSuccess) {
    cudaGetLastError();
    return fail(OCF_ERR_NOMEM, "ocf_host_alloc: cudaMallocHost(" + std::to_string(bytes) + ") failed");
  }
  return OCF_OK;
}
extern "C" int ocf_host_free(void* p) {
  if (p) cudaFreeHost(p);
  return OCF_OK;
}


// ---- optional per-kernel timing with CUDA events on the launching stream -------------------
namespace ocf {
constexpr int N_TAGS = 10;
struct Profiler {
  bool on = false;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev[N_TAGS];
  size_t used[N_TAGS] = {0};
  cudaEvent_t pending = nullptr;
  void begin(int tag, cudaStream_t st) {
    if (!on) return;
    if (used[tag] == ev[tag].size()) {
      cudaEvent_t a, b;
      cudaEventCreate(&a); cudaEventCreate(&b);
      ev[tag].push_back({a, b});
    }
    cudaEventRecord(ev[tag][used[tag]].first, st);
  }
  void end(int tag, cudaStream_t st) {
    if (!on) return;
    cudaEventRecord(ev[tag][used[tag]].second, st);
    used[tag] += 1;
  }
};
static Profiler g_prof;
}  // namespace ocf

extern "C" int ocf_profile_enable(int on) {
  g_prof.on = on != 0;
  return OCF_OK;
}
extern "C" int ocf_profile_reset(void) {
  for (int t = 0; t < N_TAGS; ++t) g_prof.used[t] = 0;
  return OCF_OK;
}
extern "C" int ocf_profile_read(int tag, double* total_ms, int64_t* count) {
  OCF_REQUIRE(tag >= 0 && tag < N_TAGS && total_ms && count, "ocf_profile_read: bad argument");
  OCF_CUDA(cudaDeviceSynchronize());
  double tot = 0.0;
  for (size_t k = 0; k < g_prof.used[tag]; ++k) {
    float ms = 0.f;
    OCF_CUDA(cudaEventElapsedTime(&ms, g_prof.ev[tag][k].first, g_prof.ev[tag][k].second));
    tot += ms;
  }
  *total_ms = tot; *count = (int64_t)g_prof.used[tag];
  return OCF_OK;
}

// ============================================================================================
// store
// ============================================================================================
extern "C" int ocf_store_create(int64_t n_rows, int64_t n_cols, const int64_t* rowptr, const int32_t* col,
                                const float* val, ocf_store** out) {
  OCF_REQUIRE(out != nullptr && rowptr != nullptr, "ocf_store_create: null argument");
  *out = nullptr;
  OCF_REQUIRE(n_rows >= 0 && n_cols > 0 && n_cols < (int64_t(1) << 31), "ocf_store_create: bad shape");
  OCF_REQUIRE(rowptr[0] == 0, "ocf_store_create: rowptr[0] must be 0");
  const int64_t nnz = rowptr[n_rows];
  OCF_REQUIRE(nnz >= 0 && nnz < (int64_t(1) << 31), "ocf_store_create: nnz must be < 2^31");
  OCF_REQUIRE(nnz == 0 || (col != nullptr && val != nullptr), "ocf_store_create: null col/val");
  for (int64_t r = 0; r < n_rows; ++r)
    OCF_REQUIRE(rowptr[r + 1] >= rowptr[r], "ocf_store_create: rowptr not monotone");
  ocf_store* s = new ocf_store();
  s->n_rows = n_rows; s->n_cols = n_cols; s->nnz = nnz;
  s->h_rowptr.assign(rowptr, rowptr + n_rows + 1);

  // repeated columns inside a row -> next_dup chains (last-write-wins resolution in K1)
  std::vector<int32_t> stamp((size_t)n_cols, -1), lastpos;
  std::vector<int32_t> next_dup;
  for (int64_t r = 0; r < n_rows && !s->has_dups; ++r)
    for (int64_t e = rowptr[r]; e < rowptr[r + 1]; ++e) {
      const int32_t c = col[e];
      if (c < 0 || c >= n_cols) { delete s; return fail(OCF_ERR_INVALID, "ocf_store_create: column out of range"); }
      if (stamp[c] == (int32_t)r) { s->has_dups = true; break; }
      stamp[c] = (int32_t)r;
    }
  if (s->has_dups) {
    next_dup.assign((size_t)nnz, -1);
    lastpos.assign((size_t)n_cols, -1);
    std::fill(stamp.begin(), stamp.end(), -1);
    for (int64_t r = 0; r < n_rows; ++r) {
      const int64_t a = rowptr[r], b = rowptr[r + 1];
      for (int64_t e = b - 1; e >= a; --e) {
        const int32_t c = col[e];
        if (c < 0 || c >= n_cols) { delete s; return fail(OCF_ERR_INVALID, "ocf_store_create: column out of range"); }
        next_dup[e] = (stamp[c] == (int32_t)r) ? lastpos[c] : -1;
        stamp[c] = (int32_t)r;
        lastpos[c] = (int32_t)(e - a);
      }
    }
  }
  int st = OCF_OK;
  int64_t* d_rowptr = nullptr; int32_t* d_col = nullptr; float* d_val = nullptr; int32_t* d_nd = nullptr;
  auto bail = [&](int code) { s->mem.release(); delete s; return code; };
  if ((st = s->mem.get(&d_rowptr, (size_t)n_rows + 1)) || (st = s->mem.get(&d_col, (size_t)nnz)) ||
      (st = s->mem.get(&d_val, (size_t)nnz)))
    return bail(st);
  if (cudaMemcpy(d_rowptr, rowptr, sizeof(int64_t) * (n_rows + 1), cudaMemcpyHostToDevice) != cudaSuccess ||
      (nnz && cudaMemcpy(d_col, col, sizeof(int32_t) * nnz, cudaMemcpyHostToDevice) != cudaSuccess) ||
      (nnz && cudaMemcpy(d_val, val, sizeof(float) * nnz, cudaMemcpyHostToDevice) != cudaSuccess))
    return bail(fail(OCF_ERR_CUDA, "ocf_store_create: upload failed"));
  if (s->has_dups) {
    if ((st = s->mem.get(&d_nd, (size_t)nnz))) return bail(st);
    if (cudaMemcpy(d_nd, next_dup.data(), sizeof(int32_t) * nnz, cudaMemcpyHostToDevice) != cudaSuccess)
      return bail(fail(OCF_ERR_CUDA, "ocf_store_create: upload failed"));
  }
  s->dev.rowptr = d_rowptr; s->dev.col = d_col; s->dev.val = d_val; s->dev.next_dup = d_nd;
  *out = s;
  return OCF_OK;
}

extern "C" int ocf_store_destroy(ocf_store* s) {
  if (s) { s->mem.release(); delete s; }
  return OCF_OK;
}

extern "C" int ocf_store_info(const ocf_store* s, int64_t info[5]) {
  OCF_REQUIRE(s && info, "ocf_store_info: null argument");
  info[0] = s->n_rows; info[1] = s->n_cols; info[2] = s->nnz; info[3] = s->has_dups ? 1 : 0;
  info[4] = (int64_t)s->mem.bytes;
  return OCF_OK;
}

extern "C" int ocf_pair_create(const ocf_store* in, const ocf_store* tg, ocf_pair** out) {
  OCF_REQUIRE(in && tg && out, "ocf_pair_create: null argument");
  *out = nullptr;
  OCF_REQUIRE(in->n_rows == tg->n_rows && in->n_cols == tg->n_cols, "ocf_pair_create: stores must have the same rows and columns");
  ocf_pair* p = new ocf_pair();
  p->in = in; p->tg = tg;
  // input ratings whose column is also a target of the same row (missing-data mask counted once)
  std::vector<int32_t> hc_in((size_t)in->nnz), hc_tg((size_t)tg->nnz);
  if (in->nnz && cudaMemcpy(hc_in.data(), in->dev.col, sizeof(int32_t) * in->nnz, cudaMemcpyDeviceToHost) != cudaSuccess) { delete p; return fail(OCF_ERR_CUDA, "ocf_pair_create: download failed"); }
  if (tg->nnz && cudaMemcpy(hc_tg.data(), tg->dev.col, sizeof(int32_t) * tg->nnz, cudaMemcpyDeviceToHost) != cudaSuccess) { delete p; return fail(OCF_ERR_CUDA, "ocf_pair_create: download failed"); }
  std::vector<int32_t> stamp((size_t)in->n_cols, -1);
  std::vector<uint8_t> ov((size_t)in->nnz, 0);
  bool any = false;
  for (int64_t r = 0; r < in->n_rows; ++r) {
    for (int64_t e = tg->h_rowptr[r]; e < tg->h_rowptr[r + 1]; ++e) stamp[hc_tg[e]] = (int32_t)r;
    for (int64_t e = in->h_rowptr[r]; e < in->h_rowptr[r + 1]; ++e)
      if (stamp[hc_in[e]] == (int32_t)r) { ov[e] = 1; any = true; }
  }
  if (any) {
    int st = p->mem.get(&p->d_in_overlap, (size_t)in->nnz);
    if (st) { delete p; return st; }
    if (cudaMemcpy(p->d_in_overlap, ov.data(), ov.size(), cudaMemcpyHostToDevice) != cudaSuccess) { p->mem.release(); delete p; return fail(OCF_ERR_CUDA, "ocf_pair_create: upload failed"); }
  }
  *out = p;
  return OCF_OK;
}

extern "C" int ocf_pair_destroy(ocf_pair* p) {
  if (p) { p->mem.release(); delete p; }
  return OCF_OK;
}

// ============================================================================================
// batch
// ============================================================================================
// Upper bound of the work items of any batch within (max_rows, max_entries): pick_chunk() keeps
// the chunk length >= ceil(entries / TARGET_ITEMS), so items <= TARGET_ITEMS + rows.
constexpr int64_t TARGET_ITEMS = 148 * 6;
static int max_items_for(int max_rows, int64_t max_entries) {
  return (int)std::min<int64_t>(max_entries / 32 + max_rows + 1, TARGET_ITEMS + max_rows + 1);
}

// Fixed for the life of a batch object (sized by its capacity), so that every device pointer a kernel
// gets is the same for every fill: [header | row_ids | ent_off | in_len | item_ptr | items | draw_off | flags].
// One copy uploads the prefix up to the flags (or through them when the host supplies the flags).
static size_t staging_layout(int max_rows, int max_items, int64_t max_entries, size_t off[8]) {
  size_t o = 0;
  off[0] = o; o = align_up(o + sizeof(BatchHdr), 64);                        // header
  off[1] = o; o = align_up(o + sizeof(int32_t) * max_rows, 16);              // row_ids
  off[2] = o; o = align_up(o + sizeof(int32_t) * (max_rows + 1), 16);        // ent_off
  off[3] = o; o = align_up(o + sizeof(int32_t) * max_rows, 16);              // in_len
  off[4] = o; o = align_up(o + sizeof(int32_t) * (max_rows + 1), 16);        // item_ptr
  off[5] = o; o = align_up(o + sizeof(int4) * (size_t)max_items, 16);        // items
  off[6] = o; o = align_up(o + sizeof(int32_t) * max_rows, 16);              // draw_off (device-RNG mode)
  off[7] = o; o = align_up(o + (size_t)max_entries, 16);                     // flags (last: not uploaded when the device derives them)
  return o;
}

static std::atomic<uint64_t> g_batch_uid{0};

extern "C" int ocf_batch_create(int32_t max_rows, int64_t max_entries, ocf_batch** out) {
  OCF_REQUIRE(out != nullptr, "ocf_batch_create: null argument");
  *out = nullptr;
  OCF_REQUIRE(max_rows > 0 && max_rows <= MAX_BATCH_ROWS, "ocf_batch_create: max_rows must be in 1..4096");
  OCF_REQUIRE(max_entries >= 0 && max_entries < (int64_t(1) << 31), "ocf_batch_create: bad max_entries");
  ocf_batch* b = new ocf_batch();
  b->max_rows = max_rows; b->max_entries = max_entries;
  b->uid = ++g_batch_uid;
  b->max_items = max_items_for(max_rows, max_entries);
  b->staging_bytes = staging_layout(max_rows, b->max_items, max_entries, b->off);
  auto bail = [&](int code) {
    b->mem.release(); if (b->h_staging) cudaFreeHost(b->h_staging); if (b->copied) cudaEventDestroy(b->copied);
    if (b->gstream) cudaStreamDestroy(b->gstream); if (b->gathered) cudaEventDestroy(b->gathered); if (b->consumed) cudaEventDestroy(b->consumed);
    if (b->wl_ready) cudaEventDestroy(b->wl_ready);
    delete b; return code; };
  if (cudaMallocHost(reinterpret_cast<void**>(&b->h_staging), b->staging_bytes) != cudaSuccess)
    return bail(fail(OCF_ERR_NOMEM, "ocf_batch_create: pinned allocation failed"));
  if (cudaEventCreateWithFlags(&b->copied, cudaEventDisableTiming) != cudaSuccess)
    return bail(fail(OCF_ERR_CUDA, "ocf_batch_create: event creation failed"));
  {
    int hi = 0;
    cudaDeviceGetStreamPriorityRange(nullptr, &hi);
    if (cudaStreamCreateWithPriority(&b->gstream, cudaStreamNonBlocking, hi) != cudaSuccess ||
        cudaEventCreateWithFlags(&b->gathered, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&b->wl_ready, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&b->consumed, cudaEventDisableTiming) != cudaSuccess)
      return bail(fail(OCF_ERR_CUDA, "ocf_batch_create: stream / event creation failed"));
  }
  int st;
  if ((st = b->mem.get(&b->d_staging, b->staging_bytes)) || (st = b->mem.get(&b->d_ent_col, (size_t)max_entries)) ||
      (st = b->mem.get(&b->d_ent_val, (size_t)max_entries)) || (st = b->mem.get(&b->d_codes, (size_t)max_entries)))
    return bail(st);
  std::memset(b->h_staging, 0, b->staging_bytes);
  BatchDev& d = b->dev;
  const size_t* off = b->off;
  d.hdr = reinterpret_cast<const BatchHdr*>(b->d_staging + off[0]);
  d.row_ids = reinterpret_cast<const int32_t*>(b->d_staging + off[1]);
  d.ent_off = reinterpret_cast<const int32_t*>(b->d_staging + off[2]);
  d.in_len = reinterpret_cast<const int32_t*>(b->d_staging + off[3]);
  d.item_ptr = reinterpret_cast<const int32_t*>(b->d_staging + off[4]);
  d.items = reinterpret_cast<const int4*>(b->d_staging + off[5]);
  d.draw_off = reinterpret_cast<const int32_t*>(b->d_staging + off[6]);
  d.flags = b->d_staging + off[7];
  d.flags_out = b->d_staging + off[7];
  d.ent_col = b->d_ent_col; d.ent_val = b->d_ent_val; d.codes = b->d_codes;
  *out = b;
  return OCF_OK;
}

extern "C" int ocf_batch_destroy(ocf_batch* b) {
  if (b) {
    if (b->gstream) { cudaStreamSynchronize(b->gstream); cudaStreamDestroy(b->gstream); }
    if (b->gathered) cudaEventDestroy(b->gathered);
    if (b->consumed) cudaEventDestroy(b->consumed);
    if (b->wl_ready) cudaEventDestroy(b->wl_ready);
    if (b->wl_graph) cudaGraphExecDestroy(b->wl_graph);
    b->wl_mem.release();
    b->mem.release();
    if (b->h_staging) cudaFreeHost(b->h_staging);
    if (b->copied) cudaEventDestroy(b->copied);
    delete b;
  }
  return OCF_OK;
}

// Work items: chunks of <= CH ratings of one row, CH sized so that the row-centric kernels get
// a few CTAs per SM whatever the batch looks like.
static int pick_chunk(int64_t n_entries) {
  int64_t ch = (n_entries + TARGET_ITEMS - 1) / TARGET_ITEMS;
  ch = (int64_t)align_up((size_t)std::max<int64_t>(ch, 1), 32);
  return (int)std::max<int64_t>(ch, 32);
}

// `draw_len` (device-RNG mode): draws each row consumes = its FULL length (a column shard passes
// them; null = the store's own row lengths); `with_draws` stages the per-row draw offsets and
// leaves the flags to the device.
static int batch_stage(ocf_batch* b, const int32_t* row_ids, int n_rows, const std::vector<int64_t>& rp_a,
                       const std::vector<int64_t>* rp_b, int64_t n_store_rows, const uint8_t* flags,
                       int64_t n_flags, cudaStream_t stream, int hdr_pass_through, float hdr_aux,
                       bool with_draws = false, const int64_t* draw_len = nullptr) {
  OCF_REQUIRE(n_rows > 0 && n_rows <= b->max_rows, "batch fill: row count exceeds the batch capacity");
  if (b->copy_pending) { OCF_CUDA(cudaEventSynchronize(b->copied)); b->copy_pending = false; }
  // pass 1: lengths
  int64_t total = 0;
  for (int r = 0; r < n_rows; ++r) {
    const int32_t row = row_ids[r];
    OCF_REQUIRE(row >= 0 && row < n_store_rows, "batch fill: row id out of range");
    total += rp_a[row + 1] - rp_a[row];
    if (rp_b) total += (*rp_b)[row + 1] - (*rp_b)[row];
  }
  OCF_REQUIRE(total <= b->max_entries, "batch fill: more ratings than the batch capacity");
  if (flags != nullptr || n_flags >= 0) OCF_REQUIRE(n_flags == total, "batch fill: n_flags must equal the total length of the listed rows");
  const int ch = pick_chunk(total);
  int64_t n_items = 0;
  for (int r = 0; r < n_rows; ++r) {
    const int32_t row = row_ids[r];
    int64_t n = rp_a[row + 1] - rp_a[row];
    if (rp_b) n += (*rp_b)[row + 1] - (*rp_b)[row];
    n_items += std::max<int64_t>(1, (n + ch - 1) / ch);          // an empty row still gets one (empty) item: its row tail
  }
  OCF_REQUIRE(n_items <= b->max_items, "batch fill: too many work items");
  const size_t* off = b->off;
  const size_t bytes = flags != nullptr ? off[7] + (size_t)total : off[7];       // without host flags the flag slot is not copied
  uint8_t* hs = b->h_staging;
  BatchHdr* h_hdr = reinterpret_cast<BatchHdr*>(hs + off[0]);
  int32_t* h_rows = reinterpret_cast<int32_t*>(hs + off[1]);
  int32_t* h_eoff = reinterpret_cast<int32_t*>(hs + off[2]);
  int32_t* h_inlen = reinterpret_cast<int32_t*>(hs + off[3]);
  int32_t* h_iptr = reinterpret_cast<int32_t*>(hs + off[4]);
  int4* h_items = reinterpret_cast<int4*>(hs + off[5]);
  int32_t* h_draw = reinterpret_cast<int32_t*>(hs + off[6]);
  int64_t e = 0; int it = 0; int64_t tcount = 0; int64_t draw = b->draw_base;   // the sparsity draws come first
  for (int r = 0; r < n_rows; ++r) {
    const int32_t row = row_ids[r];
    const int64_t na = rp_a[row + 1] - rp_a[row];
    const int64_t nb = rp_b ? (*rp_b)[row + 1] - (*rp_b)[row] : 0;
    h_rows[r] = row; h_eoff[r] = (int32_t)e; h_inlen[r] = (int32_t)na; h_iptr[r] = it;
    if (with_draws) { h_draw[r] = (int32_t)draw; draw += draw_len ? draw_len[r] : na; }
    const int64_t n = na + nb;
    // item = (batch row, start inside the row, length, absolute position of the first entry)
    if (n == 0) h_items[it++] = make_int4(r, 0, 0, (int)e);
    for (int64_t s0 = 0; s0 < n; s0 += ch) h_items[it++] = make_int4(r, (int)s0, (int)std::min<int64_t>(ch, n - s0), (int)(e + s0));
    e += n; tcount += nb;
  }
  h_eoff[n_rows] = (int32_t)e; h_iptr[n_rows] = it;
  h_hdr->B = n_rows; h_hdr->n_items = (int)n_items; h_hdr->n_entries = (int)total;
  h_hdr->cdf_row0 = b->cdf0_row0; h_hdr->pass_through = hdr_pass_through;
  h_hdr->rng_lo = b->rng_lo; h_hdr->rng_range = b->rng_range; h_hdr->aux_value = hdr_aux;
  h_hdr->word_base = b->word_base; h_hdr->ring_words = b->ring_words;
  if (flags != nullptr && total > 0) std::memcpy(hs + off[7], flags, (size_t)total);
  OCF_CUDA(cudaMemcpyAsync(b->d_staging, hs, bytes, cudaMemcpyHostToDevice, stream));
  OCF_CUDA(cudaEventRecord(b->copied, stream));
  b->copy_pending = true;
  b->last_h2d = bytes;
  b->target_count = tcount;
  BatchDev& d = b->dev;
  d.B = n_rows; d.n_items = (int)n_items; d.n_entries = (int)total;
  d.words = b->d_words; d.rng_lo = b->rng_lo; d.rng_range = b->rng_range; d.cdf_row0 = b->cdf0_row0;
  return OCF_OK;
}

// K1 on the row ids / flags already resident in the batch's device staging.
static int launch_gather(ocf_batch* b, cudaStream_t stream) {
  if (b->dev.n_items == 0) return OCF_OK;
  g_prof.begin(0, stream);
  if (b->mode == 1 && b->rng_mode) k_gather_split<true><<<b->dev.n_items, 128, 0, stream>>>(b->store->dev, b->dev);
  else if (b->mode == 1) k_gather_split<false><<<b->dev.n_items, 128, 0, stream>>>(b->store->dev, b->dev);
  else k_gather_fixed<<<b->dev.n_items, 128, 0, stream>>>(b->pair->in->dev, b->pair->tg->dev, b->pair->d_in_overlap, b->dev);
  OCF_LAUNCHED();
  g_prof.end(0, stream);
  return OCF_OK;
}

// The stream a fill of `b` runs on, ordered after the last consumer of the batch's tiles.
static cudaStream_t fill_begin(ocf_batch* b) {
  if (b->consumed_valid) cudaStreamWaitEvent(b->gstream, b->consumed, 0);
  return b->gstream;
}
static int fill_end(ocf_batch* b, cudaStream_t user, cudaStream_t used) {
  b->fill_seq += 1;               // a work list built for an earlier fill is stale
  b->gathered_valid = false;
  if (used != user) { OCF_CUDA(cudaEventRecord(b->gathered, used)); b->gathered_valid = true; }
  return OCF_OK;
}
// Consumers of a batch's tiles (steps, predict / score, densify, flag read-back) on stream `st`.
static int batch_acquire(const ocf_batch* b, cudaStream_t st) {
  if (b->gathered_valid) OCF_CUDA(cudaStreamWaitEvent(st, b->gathered, 0));
  return OCF_OK;
}
static int batch_release(const ocf_batch* cb, cudaStream_t st) {
  ocf_batch* b = const_cast<ocf_batch*>(cb);
  OCF_CUDA(cudaEventRecord(b->consumed, st));
  b->consumed_valid = true;
  return OCF_OK;
}

// Caller input check of the split fills: a batch lists every row at most once.
static int check_distinct_rows(const int32_t* row_ids, int32_t n_rows, const char* who) {
  std::vector<int32_t> tmp(row_ids, row_ids + std::max(n_rows, 0));
  std::sort(tmp.begin(), tmp.end());
  if (std::adjacent_find(tmp.begin(), tmp.end()) != tmp.end()) return fail(OCF_ERR_INVALID, std::string(who) + ": a row appears twice in the batch");
  return OCF_OK;
}

extern "C" int ocf_batch_fill_split(ocf_batch* b, const ocf_store* store, const int32_t* row_ids, int32_t n_rows,
                                    const uint8_t* keep_flags, int64_t n_flags, int pass_through,
                                    float aux_var_value, void* stream_) {
  OCF_REQUIRE(b && store && row_ids, "ocf_batch_fill_split: null argument");
  OCF_REQUIRE(keep_flags != nullptr || n_flags == 0, "ocf_batch_fill_split: null keep_flags");
  cudaStream_t user = as_stream(stream_);
  cudaStream_t stream = fill_begin(b);
  OCF_TRY(check_distinct_rows(row_ids, n_rows, "ocf_batch_fill_split"));
  OCF_TRY(batch_stage(b, row_ids, n_rows, store->h_rowptr, nullptr, store->n_rows, keep_flags, n_flags, stream,
                      pass_through ? 1 : 0, aux_var_value));
  b->mode = 1; b->store = store; b->aux_value = aux_var_value; b->rng_mode = false;
  // in split mode every listed rating is a target when pass_through, else the flag-0 ones
  int64_t tc = 0;
  if (pass_through) tc = n_flags; else for (int64_t k = 0; k < n_flags; ++k) tc += keep_flags[k] == 0;
  b->target_count = tc;
  b->pass_through = pass_through ? 1 : 0;
  OCF_TRY(launch_gather(b, stream));
  return fill_end(b, user, stream);
}

extern "C" int ocf_batch_fill_split_uniform(ocf_batch* b, const ocf_store* store, const int32_t* row_ids, int32_t n_rows,
                                            const double* u, int64_t n_u, const double* cdf0, const int32_t* orig_pos,
                                            const int64_t* full_len, int pass_through, float aux_var_value, void* stream_) {
  OCF_REQUIRE(b && store && row_ids && cdf0 && (u || n_u == 0), "ocf_batch_fill_split_uniform: null argument");
  OCF_REQUIRE(n_rows > 0 && n_rows <= b->max_rows, "ocf_batch_fill_split_uniform: row count exceeds the batch capacity");
  // keep flag of a rating = (its uniform draw >= cdf0 of its row): exactly what
  // np.random.choice([0,1], n, p=[1-s, s]) returns for that draw (data_reader.py:130)
  std::vector<uint8_t>& flags = b->flag_scratch;
  int64_t total = 0, full_total = 0;
  for (int r = 0; r < n_rows; ++r) {
    const int32_t row = row_ids[r];
    OCF_REQUIRE(row >= 0 && row < store->n_rows, "ocf_batch_fill_split_uniform: row id out of range");
    total += store->h_rowptr[row + 1] - store->h_rowptr[row];
    full_total += full_len ? full_len[r] : store->h_rowptr[row + 1] - store->h_rowptr[row];
  }
  OCF_REQUIRE(full_total == n_u, "ocf_batch_fill_split_uniform: n_u must equal the total (full) length of the listed rows");
  flags.resize((size_t)total);
  int64_t k = 0, off = 0;
  for (int r = 0; r < n_rows; ++r) {
    const int32_t row = row_ids[r];
    const int64_t e0 = store->h_rowptr[row], n = store->h_rowptr[row + 1] - e0;
    const double c0 = cdf0[r];
    const double* ur = u + off;
    if (orig_pos) for (int64_t j = 0; j < n; ++j) flags[k++] = ur[orig_pos[e0 + j]] >= c0;
    else for (int64_t j = 0; j < n; ++j) flags[k++] = ur[j] >= c0;
    off += full_len ? full_len[r] : n;
  }
  return ocf_batch_fill_split(b, store, row_ids, n_rows, flags.data(), total, pass_through, aux_var_value, stream_);
}

extern "C" int ocf_batch_fill_fixed(ocf_batch* b, const ocf_pair* pair, const int32_t* row_ids, int32_t n_rows,
                                    float aux_var_value, void* stream_) {
  OCF_REQUIRE(b && pair && row_ids, "ocf_batch_fill_fixed: null argument");
  cudaStream_t user = as_stream(stream_);
  cudaStream_t stream = fill_begin(b);
  OCF_TRY(batch_stage(b, row_ids, n_rows, pair->in->h_rowptr, &pair->tg->h_rowptr, pair->in->n_rows, nullptr, -1, stream,
                      0, aux_var_value));
  b->mode = 2; b->store = pair->tg; b->aux_value = aux_var_value;
  b->pair = pair;
  OCF_TRY(launch_gather(b, stream));
  return fill_end(b, user, stream);
}

extern "C" int ocf_batch_regather(ocf_batch* b, void* stream_) {
  OCF_REQUIRE(b, "ocf_batch_regather: null argument");
  if (b->mode == 0) return fail(OCF_ERR_STATE, "ocf_batch_regather: the batch has not been filled");
  b->rng_mode = false;            // the first gather left the flags in the device staging
  cudaStream_t user = as_stream(stream_);
  // A re-gather has no host copy to hide. On its own stream it still overlaps the previous step (Jester: 71 -> 66 us per
  // step), but beside a step that holds NCCL collectives it costs more than it hides (2 GPUs: 785 vs 855 M ratings/s),
  // so a process with a communicator keeps it on the caller's stream.
  const bool regather_sync = g_comms_alive.load() > 0;
  cudaStream_t stream = regather_sync ? user : fill_begin(b);
  if (regather_sync) OCF_TRY(batch_acquire(b, user));
  if (stream != user && b->gathered_valid) OCF_CUDA(cudaStreamWaitEvent(stream, b->gathered, 0));   // same stream: already in order
  OCF_TRY(launch_gather(b, stream));
  return fill_end(b, user, stream);
}

// ---- NumPy MT19937 on the device ------------------------------------------------------------------
static void rng_release(ocf_rng* r) {
  for (cudaStream_t st : r->wstream) { cudaStreamSynchronize(st); cudaStreamDestroy(st); }
  for (cudaEvent_t e : r->block_ev) cudaEventDestroy(e);
  for (cudaEvent_t e : r->slot_free) cudaEventDestroy(e);
  if (r->placed) cudaEventDestroy(r->placed);
  if (r->io) { cudaStreamDestroy(r->io); r->io = nullptr; }
  r->wstream.clear(); r->block_ev.clear(); r->slot_free.clear(); r->placed = nullptr;
  r->mem.release();
  r->d_ring = r->d_arrays = r->d_seq = r->d_poly = nullptr;
}

// (Re)builds the service: `workers` generator CTAs, blocks of `block_regens` regenerations, a ring of at least
// `ring_words_min` words. Drops whatever stream state the object held (set_state must follow).
static int rng_setup(ocf_rng* r, int workers, int block_regens, int64_t ring_words_min) {
  OCF_REQUIRE(workers >= 1 && workers <= 32 && block_regens >= 1 && block_regens <= (1 << 16), "ocf_rng_configure: workers must be 1..32, block_regens 1..65536");
  OCF_CUDA(cudaSetDevice(r->device));
  rng_release(r);
  r->M = workers; r->C = block_regens;
  r->BW = (int64_t)block_regens * 624;
  // room for the batch being read, the batch being generated and every worker's block in flight
  const int64_t want = std::max<int64_t>(ring_words_min, 4 * r->BW) + (int64_t)(2 * workers + 2) * r->BW;
  r->R = (int)((want + r->BW - 1) / r->BW);
  r->RW = (int64_t)r->R * r->BW;
  OCF_REQUIRE(r->RW < (int64_t(1) << 31), "ocf_rng_configure: ring too large");
  if (workers > 1) {
    OCF_REQUIRE(mtj::phi_ok(), "ocf_rng_configure: could not recover MT19937's characteristic polynomial");
    uint32_t poly[2][624];
    mtj::to_words(mtj::x_pow((uint64_t)r->BW), poly[0]);
    mtj::to_words(mtj::x_pow((uint64_t)r->BW * (uint64_t)(workers - 1)), poly[1]);
    OCF_TRY(r->mem.get(&r->d_poly, 2 * 624));
    OCF_CUDA(cudaMemcpy(r->d_poly, poly, sizeof(poly), cudaMemcpyHostToDevice));
    OCF_TRY(r->mem.get(&r->d_seq, (size_t)workers * MT_SEQ_REGENS * 624));
  }
  OCF_TRY(r->mem.get(&r->d_ring, (size_t)r->RW));
  OCF_TRY(r->mem.get(&r->d_arrays, (size_t)workers * 2 * 640, true));
  r->wstream.resize(workers); r->cur.assign(workers, 0);
  for (int j = 0; j < workers; ++j) OCF_CUDA(cudaStreamCreateWithFlags(&r->wstream[j], cudaStreamNonBlocking));
  r->block_ev.resize(r->R); r->slot_free.resize(r->R); r->slot_free_valid.assign(r->R, 0);
  for (int k = 0; k < r->R; ++k) {
    OCF_CUDA(cudaEventCreateWithFlags(&r->block_ev[k], cudaEventDisableTiming));
    OCF_CUDA(cudaEventCreateWithFlags(&r->slot_free[k], cudaEventDisableTiming));
  }
  OCF_CUDA(cudaEventCreateWithFlags(&r->placed, cudaEventDisableTiming));
  r->have_state = false; r->next_block = 0; r->pos_u = 0;
  return OCF_OK;
}

extern "C" int ocf_rng_create(ocf_rng** out) {
  OCF_REQUIRE(out != nullptr, "ocf_rng_create: null argument");
  *out = nullptr;
  ocf_rng* r = new ocf_rng();
  if (cudaGetDevice(&r->device) != cudaSuccess) { cudaGetLastError(); delete r; return fail(OCF_ERR_CUDA, "ocf_rng_create: no CUDA device"); }
  int workers = 2;
  if (const char* e = std::getenv("OCF_RNG_WORKERS")) workers = std::max(1, std::min(32, std::atoi(e)));
  const int st = rng_setup(r, workers, 256, 0);
  if (st) { rng_release(r); delete r; return st; }
  *out = r;
  return OCF_OK;
}

extern "C" int ocf_rng_configure(ocf_rng* r, int32_t workers, int32_t block_regens, int64_t ring_words_min) {
  OCF_REQUIRE(r != nullptr, "ocf_rng_configure: null argument");
  if (workers <= 0) workers = r->M;
  if (block_regens <= 0) block_regens = r->C;
  // nothing to do when the current ring already satisfies the request
  if (workers == r->M && block_regens == r->C && std::max<int64_t>(ring_words_min, 4 * r->BW) + (int64_t)(2 * workers + 2) * r->BW <= r->RW)
    return OCF_OK;
  uint32_t key[624]; int32_t pos = 0;
  const bool keep = r->have_state;
  if (keep) OCF_TRY(ocf_rng_get_state(r, key, &pos));
  OCF_TRY(rng_setup(r, workers, block_regens, ring_words_min));
  if (keep) OCF_TRY(ocf_rng_set_state(r, key, pos));
  return OCF_OK;
}

extern "C" int ocf_rng_info(const ocf_rng* r, int64_t info[6]) {
  OCF_REQUIRE(r && info, "ocf_rng_info: null argument");
  info[0] = r->M; info[1] = r->C; info[2] = r->R; info[3] = r->RW; info[4] = r->pos_u; info[5] = r->next_block;
  return OCF_OK;
}

extern "C" int ocf_rng_destroy(ocf_rng* r) {
  if (r) { cudaSetDevice(r->device); rng_release(r); delete r; }
  return OCF_OK;
}

// array `src` of worker j jumped by polynomial `which` into its other buffer, on stream st
static int rng_jump(ocf_rng* r, int j, const uint32_t* src, uint32_t* dst, int which, cudaStream_t st) {
  uint32_t* seq = r->d_seq + (size_t)j * MT_SEQ_REGENS * 624;
  // the worker's own sequence from `src` on (src itself stays as it is), dst zeroed for the XOR accumulation
  k_mt_block<false><<<1, MT_THREADS, 0, st>>>(dst, MT_SEQ_REGENS - 1, seq, (uint32_t)(MT_SEQ_REGENS * 624), 624u, src, dst);
  OCF_LAUNCHED();
  k_mt_jump_apply<<<MT_JUMP_CTAS, MT_THREADS, 0, st>>>(seq, r->d_poly + (size_t)which * 624, dst);
  OCF_LAUNCHED();
  return OCF_OK;
}

extern "C" int ocf_rng_set_state(ocf_rng* r, const uint32_t* key, int32_t pos) {
  OCF_REQUIRE(r && key && pos >= 0 && pos <= 624, "ocf_rng_set_state: bad argument");
  OCF_CUDA(cudaSetDevice(r->device));        // generator threads call this too
  for (cudaStream_t st : r->wstream) OCF_CUDA(cudaStreamSynchronize(st));
  std::memcpy(r->origin, key, sizeof(r->origin));
  r->pos_u = pos; r->next_block = 0; r->have_state = true;
  std::fill(r->slot_free_valid.begin(), r->slot_free_valid.end(), 0);
  std::fill(r->cur.begin(), r->cur.end(), 0);
  // the origin array's own (tempered) words are stream words 0..623
  uint32_t tempered[624];
  for (int i = 0; i < 624; ++i) tempered[i] = mtj::temper(key[i]);
  cudaStream_t s0 = r->wstream[0];
  OCF_CUDA(cudaMemcpyAsync(r->d_ring, tempered, sizeof(tempered), cudaMemcpyHostToDevice, s0));
  OCF_CUDA(cudaMemcpyAsync(r->array_of(0, 0), key, 624 * sizeof(uint32_t), cudaMemcpyHostToDevice, s0));
  // worker j starts C regenerations after worker j - 1
  for (int j = 1; j < r->M; ++j) OCF_TRY(rng_jump(r, j, r->array_of(j - 1, 0), r->array_of(j, 0), 0, s0));
  OCF_CUDA(cudaStreamSynchronize(s0));       // `tempered` / `key` are stack / caller memory
  return OCF_OK;
}

// Enqueues the generation of every block up to `upto` (inclusive) that the ring has room for. A block's slot is
// reused once the consumers have read past the block that last lived in it.
static int rng_enqueue_blocks(ocf_rng* r, int64_t upto) {
  while (r->next_block <= upto) {
    const int64_t k = r->next_block;
    const int64_t evicted_end = 624 + (k - r->R + 1) * r->BW;       // end of the block this one overwrites
    if (k >= r->R && evicted_end > r->pos_u) break;                 // its words are not consumed yet
    const int j = (int)(k % r->M), slot = (int)(k % r->R);
    cudaStream_t st = r->wstream[j];
    if (r->slot_free_valid[slot]) OCF_CUDA(cudaStreamWaitEvent(st, r->slot_free[slot], 0));
    uint32_t* arr = r->array_of(j, r->cur[j]);
    const uint32_t off = (uint32_t)((624 + k * r->BW) % r->RW);
    k_mt_block<true><<<1, MT_THREADS, 0, st>>>(arr, r->C, r->d_ring, (uint32_t)r->RW, off);
    OCF_LAUNCHED();
    OCF_CUDA(cudaEventRecord(r->block_ev[slot], st));
    if (r->M > 1) {                                                 // over the other workers' blocks
      OCF_TRY(rng_jump(r, j, arr, r->array_of(j, r->cur[j] ^ 1), 1, st));
      r->cur[j] ^= 1;
    }
    r->last_worker = j;
    r->next_block += 1;
  }
  return OCF_OK;
}

static inline int64_t rng_block_of(const ocf_rng* r, int64_t u) { return u < 624 ? -1 : (u - 624) / r->BW; }

extern "C" int ocf_rng_prefetch(ocf_rng* r, int64_t n_draws) {
  OCF_REQUIRE(r && n_draws >= 0, "ocf_rng_prefetch: bad argument");
  if (!r->have_state) return fail(OCF_ERR_STATE, "ocf_rng_prefetch: no stream state (ocf_rng_set_state first)");
  OCF_CUDA(cudaSetDevice(r->device));
  return rng_enqueue_blocks(r, rng_block_of(r, r->pos_u + 2 * n_draws));
}

extern "C" int ocf_rng_get_state(ocf_rng* r, uint32_t* key, int32_t* pos) {
  OCF_REQUIRE(r && key && pos, "ocf_rng_get_state: null argument");
  if (!r->have_state) return fail(OCF_ERR_STATE, "ocf_rng_get_state: no stream state");
  OCF_CUDA(cudaSetDevice(r->device));
  int64_t g = r->pos_u / 624;
  int32_t p = (int32_t)(r->pos_u % 624);
  if (p == 0 && g > 0) { g -= 1; p = 624; }          // NumPy regenerates lazily: "array g - 1, exhausted"
  *pos = p;
  if (g == 0) { std::memcpy(key, r->origin, sizeof(r->origin)); return OCF_OK; }
  const int64_t k = (g - 1) / r->C;                  // the block regeneration g lives in
  OCF_TRY(rng_enqueue_blocks(r, k));
  if (r->next_block <= k) return fail(OCF_ERR_STATE, "ocf_rng_get_state: the stream position lies beyond the ring");
  const int slot = (int)(k % r->R);
  OCF_CUDA(cudaEventSynchronize(r->block_ev[slot]));
  uint32_t tmp[624];
  // the block is complete (event above); a synchronous copy would also wait for every train step queued on the legacy
  // stream and drain the pipeline at each epoch boundary (the host needs the state for np.random.permutation)
  if (r->io == nullptr) OCF_CUDA(cudaStreamCreateWithFlags(&r->io, cudaStreamNonBlocking));
  OCF_CUDA(cudaMemcpyAsync(tmp, r->d_ring + (size_t)((624 * g) % r->RW), sizeof(tmp), cudaMemcpyDeviceToHost, r->io));
  OCF_CUDA(cudaStreamSynchronize(r->io));
  for (int i = 0; i < 624; ++i) key[i] = mtj::untemper(tmp[i]);
  return OCF_OK;
}

extern "C" int ocf_rng_last_timing(ocf_rng* r, int64_t* sm_cycles, int64_t* nanoseconds) {
  OCF_REQUIRE(r && sm_cycles && nanoseconds, "ocf_rng_last_timing: null argument");
  OCF_CUDA(cudaSetDevice(r->device));
  for (cudaStream_t st : r->wstream) OCF_CUDA(cudaStreamSynchronize(st));
  // a worker's timing words sit in the buffer its last block kernel ran on
  const int j = r->last_worker;
  uint32_t tmp[4];
  const int which = r->M > 1 ? r->cur[j] ^ 1 : r->cur[j];
  OCF_CUDA(cudaMemcpy(tmp, r->array_of(j, which) + 626, sizeof(tmp), cudaMemcpyDeviceToHost));
  *sm_cycles = (int64_t)(((uint64_t)tmp[1] << 32) | tmp[0]);
  *nanoseconds = (int64_t)(((uint64_t)tmp[3] << 32) | tmp[2]);
  return OCF_OK;
}

extern "C" int ocf_rng_skip(ocf_rng* r, int64_t n_draws) {
  OCF_REQUIRE(r && n_draws >= 0, "ocf_rng_skip: bad argument");
  if (!r->have_state) return fail(OCF_ERR_STATE, "ocf_rng_skip: no stream state");
  r->pos_u += 2 * n_draws;                           // positions only: the workers produce every block anyway
  return OCF_OK;
}

// host-side helpers of the jump (tests pin the polynomial arithmetic against NumPy without a GPU)
extern "C" int ocf_mt_jump_poly(int64_t n_words, uint32_t* poly624) {
  OCF_REQUIRE(n_words >= 0 && poly624, "ocf_mt_jump_poly: bad argument");
  OCF_REQUIRE(mtj::phi_ok(), "ocf_mt_jump_poly: could not recover MT19937's characteristic polynomial");
  mtj::to_words(mtj::x_pow((uint64_t)n_words), poly624);
  return OCF_OK;
}
extern "C" int ocf_mt_jump_apply_host(const uint32_t* key624, const uint32_t* poly624, uint32_t* out624) {
  OCF_REQUIRE(key624 && poly624 && out624, "ocf_mt_jump_apply_host: null argument");
  mtj::apply_host(key624, poly624, out624);
  return OCF_OK;
}

extern "C" int ocf_store_set_orig_pos(ocf_store* s, const int32_t* orig_pos) {
  OCF_REQUIRE(s && (orig_pos || s->nnz == 0), "ocf_store_set_orig_pos: null argument");
  int32_t* d = nullptr;
  OCF_TRY(s->mem.get(&d, (size_t)s->nnz));
  if (s->nnz) OCF_CUDA(cudaMemcpy(d, orig_pos, sizeof(int32_t) * s->nnz, cudaMemcpyHostToDevice));
  s->dev.orig_pos = d;
  return OCF_OK;
}

extern "C" int ocf_batch_fill_split_rng(ocf_batch* b, const ocf_store* store, const int32_t* row_ids, int32_t n_rows,
                                        ocf_rng* rng, double lo, double hi, const int64_t* full_len, int pass_through,
                                        float aux_var_value, const ocf_rng_slice* slice, void* stream_) {
  OCF_REQUIRE(b && store && row_ids && rng, "ocf_batch_fill_split_rng: null argument");
  OCF_REQUIRE(n_rows > 0 && n_rows <= b->max_rows, "ocf_batch_fill_split_rng: row count exceeds the batch capacity");
  OCF_REQUIRE((full_len != nullptr) == (store->dev.orig_pos != nullptr), "ocf_batch_fill_split_rng: full_len goes with a store that has ocf_store_set_orig_pos");
  cudaStream_t user = as_stream(stream_);
  cudaStream_t stream = fill_begin(b);
  int64_t draws = n_rows;
  for (int r = 0; r < n_rows; ++r) {
    const int32_t row = row_ids[r];
    OCF_REQUIRE(row >= 0 && row < store->n_rows, "ocf_batch_fill_split_rng: row id out of range");
    draws += full_len ? full_len[r] : store->h_rowptr[row + 1] - store->h_rowptr[row];
  }
  b->draw_base = n_rows; b->cdf0_row0 = 0;
  if (slice != nullptr) {
    // these rows are a slice of a larger drawing unit (a rank's rows of a global batch): the unit's
    // sparsity draws come first, then the draws of the rows before this slice
    OCF_REQUIRE(slice->n_draw_rows >= n_rows && slice->row0 >= 0 && slice->row0 + n_rows <= slice->n_draw_rows &&
                slice->draws_before >= 0 && slice->draws_total >= slice->n_draw_rows + slice->draws_before + (draws - n_rows),
                "ocf_batch_fill_split_rng: inconsistent slice");
    b->draw_base = slice->n_draw_rows + slice->draws_before;
    b->cdf0_row0 = slice->row0;
    draws = slice->draws_total;
  }
  OCF_REQUIRE(draws < (int64_t(1) << 30), "ocf_batch_fill_split_rng: too many draws in one batch");
  if (!rng->have_state) return fail(OCF_ERR_STATE, "ocf_batch_fill_split_rng: the generator has no stream state (ocf_rng_set_state first)");
  OCF_CUDA(cudaSetDevice(rng->device));
  b->rng_lo = lo; b->rng_range = hi - lo;
  // this batch's words are [u0, u1) of the stream; grow the ring if one batch does not fit it comfortably
  if (4 * draws + (int64_t)(2 * rng->M + 2) * rng->BW > rng->RW) OCF_TRY(ocf_rng_configure(rng, rng->M, rng->C, 6 * draws));
  const int64_t u0 = rng->pos_u, u1 = u0 + 2 * draws;
  const int64_t kb0 = rng_block_of(rng, u0), kb1 = rng_block_of(rng, u1 - 1);
  OCF_TRY(rng_enqueue_blocks(rng, kb1));
  if (rng->next_block <= kb1) return fail(OCF_ERR_STATE, "ocf_batch_fill_split_rng: the stream ring is too small for this batch");
  b->d_words = rng->d_ring; b->word_base = (uint32_t)(u0 % rng->RW); b->ring_words = (uint32_t)rng->RW;
  OCF_TRY(check_distinct_rows(row_ids, n_rows, "ocf_batch_fill_split_rng"));
  OCF_TRY(batch_stage(b, row_ids, n_rows, store->h_rowptr, nullptr, store->n_rows, nullptr, -1, stream,
                      pass_through ? 1 : 0, aux_var_value, true, full_len));
  b->mode = 1; b->store = store; b->aux_value = aux_var_value; b->rng_mode = true;
  b->pass_through = pass_through ? 1 : 0;
  b->target_count = pass_through ? b->dev.n_entries : -1;      // the flags never visit the host
  // the gather waits for the blocks it reads; the ring slots it read are free again once it has run
  for (int64_t k = std::max<int64_t>(kb0, 0); k <= kb1; ++k) OCF_CUDA(cudaStreamWaitEvent(stream, rng->block_ev[k % rng->R], 0));
  OCF_TRY(launch_gather(b, stream));
  for (int64_t k = std::max<int64_t>(kb0, 0); k <= kb1; ++k) {
    OCF_CUDA(cudaEventRecord(rng->slot_free[k % rng->R], stream));
    rng->slot_free_valid[k % rng->R] = 1;
  }
  rng->pos_u = u1;
  // keep the workers one round of blocks ahead of the consumers
  OCF_TRY(rng_enqueue_blocks(rng, kb1 + rng->M));
  return fill_end(b, user, stream);
}

extern "C" int ocf_batch_read_flags(ocf_batch* b, uint8_t* out, int64_t count, void* stream_) {
  OCF_REQUIRE(b && (out || count == 0), "ocf_batch_read_flags: null argument");
  if (b->mode != 1) return fail(OCF_ERR_STATE, "ocf_batch_read_flags: not a split batch");
  OCF_REQUIRE(count == b->dev.n_entries, "ocf_batch_read_flags: count must equal the batch's entries");
  cudaStream_t stream = as_stream(stream_);
  OCF_TRY(batch_acquire(b, stream));
  if (count) OCF_CUDA(cudaMemcpyAsync(out, b->dev.flags, (size_t)count, cudaMemcpyDeviceToHost, stream));
  OCF_CUDA(cudaStreamSynchronize(stream));
  return OCF_OK;
}

extern "C" int ocf_batch_info(const ocf_batch* b, int64_t info[5]) {
  OCF_REQUIRE(b && info, "ocf_batch_info: null argument");
  info[0] = b->dev.B; info[1] = b->dev.n_entries; info[2] = b->dev.n_items; info[3] = b->target_count;
  info[4] = (int64_t)b->last_h2d;
  return OCF_OK;
}

extern "C" int ocf_batch_densify(const ocf_batch* b, int which, double* out, void* stream_) {
  OCF_REQUIRE(b && out, "ocf_batch_densify: null argument");
  OCF_REQUIRE(b->mode != 0, "ocf_batch_densify: batch is empty");
  OCF_REQUIRE(which >= 0 && which <= 4, "ocf_batch_densify: which must be 0..4");
  cudaStream_t stream = as_stream(stream_);
  const int64_t n_cols = b->store->n_cols;
  const size_t count = (size_t)b->dev.B * (size_t)n_cols;
  double* d_out = nullptr;
  OCF_CUDA(cudaMalloc(reinterpret_cast<void**>(&d_out), count * sizeof(double)));
  cudaError_t e = b->gathered_valid ? cudaStreamWaitEvent(stream, b->gathered, 0) : cudaSuccess;
  if (e == cudaSuccess) e = cudaMemsetAsync(d_out, 0, count * sizeof(double), stream);
  if (e == cudaSuccess && b->dev.n_entries > 0) {
    k_densify<<<(b->dev.n_entries + 255) / 256, 256, 0, stream>>>(b->dev, which, (double)b->aux_value, (int)n_cols, d_out);
    g_launches.fetch_add(1);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaMemcpyAsync(out, d_out, count * sizeof(double), cudaMemcpyDeviceToHost, stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
  cudaFree(d_out);
  if (e != cudaSuccess) return fail(OCF_ERR_CUDA, std::string("ocf_batch_densify: ") + cudaGetErrorString(e));
  return OCF_OK;
}

// ============================================================================================
// model
// ============================================================================================
static void aux_bits(int aux, int& nblk, int3& bits) {
  bits = make_int3(CODE_IN, 0, 0);
  nblk = 1;
  switch (aux) {
    case OCF_AUX_CAUSAL: nblk = 2; bits.y = CODE_OBS; break;
    case OCF_AUX_DROPOUT: nblk = 2; bits.y = CODE_IN; break;
    case OCF_AUX_ZEROS: nblk = 2; bits.y = 0; break;
    case OCF_AUX_BOTH: nblk = 3; bits.y = CODE_IN; bits.z = CODE_OBS; break;
    default: break;
  }
}

// Batch-sized buffers (activations, work-item partials, per-entry gradients).
static int alloc_workspace(ocf_model* m, int max_rows, int64_t max_entries) {
  drop_graphs(m);
  m->ws_mem.release();
  m->dense_mem.release();
  m->dense_out = nullptr;
  m->topk_cols = nullptr; m->topk_scores = nullptr; m->topk_cap = 0;
  m->rank_ok = false;
  m->cfg.max_rows = max_rows;
  m->cfg.max_entries = max_entries;
  m->max_items = max_items_for(max_rows, max_entries);
  const int L = m->L;
  m->act_rows = (long long)align_up((size_t)max_rows, 256);   // whole TMA boxes of the scoring GEMM
  m->map_h_ok = false;
  m->zsum.assign(L, nullptr); m->act.assign(L, nullptr); m->h.assign(L, nullptr);
  m->dscale.assign(L, nullptr); m->dz.assign(L, nullptr);
  const bool drop = m->cfg.dropout_p > 0.f;
  Arena& ws = m->ws_mem;
  for (int l = 0; l < L; ++l) {
    const size_t n = (size_t)max_rows * m->hp[l];
    OCF_TRY(ws.get(&m->zsum[l], n, true));
    OCF_TRY(ws.get(&m->act[l], (size_t)m->act_rows * m->hp[l], true));
    OCF_TRY(ws.get(&m->dz[l], n, true));
    if (drop) { OCF_TRY(ws.get(&m->h[l], n, true)); OCF_TRY(ws.get(&m->dscale[l], n, true)); }
    else m->h[l] = m->act[l];
  }
  OCF_TRY(ws.get(&m->P1, (size_t)m->max_items * m->hp[0]));
  OCF_TRY(ws.get(&m->P2, (size_t)m->max_items * m->hp[L - 1]));
  OCF_TRY(ws.get(&m->itemstats, (size_t)m->max_items * ROWSTAT_W));
  {
    int hpmax = 0;
    for (int l = 0; l < L; ++l) hpmax = std::max(hpmax, m->hp[l]);
    float* G = nullptr;
    OCF_TRY(ws.get(&G, (size_t)m->max_items * hpmax));
    m->tail.G = reinterpret_cast<float4*>(G);
    OCF_TRY(ws.get(&m->tail.Gs, (size_t)m->max_items * ROWSTAT_W));
    OCF_TRY(ws.get(&m->tail.tick_grp, (size_t)m->max_items, true));      // self-resetting arrival counters
    OCF_TRY(ws.get(&m->tail.tick_row, (size_t)max_rows, true));
  }
  OCF_TRY(ws.get(&m->dy, (size_t)max_entries, true));
  // [row statistics | dL/dh of the top hidden layer] share one allocation: a column shard
  // all-reduces both with a single collective over the prefix 4*max_rows + B*hp floats
  OCF_TRY(ws.get(&m->rowstats, (size_t)max_rows * ROWSTAT_W + (size_t)max_rows * m->hp[L - 1], true));
  m->dh_top = m->rowstats + (size_t)max_rows * ROWSTAT_W;
  OCF_TRY(ws.get(&m->col_matches, (size_t)max_entries * 3));
  m->col_bits_words = (size_t)m->cfg.n_cols * (size_t)((max_rows + 31) / 32);
  OCF_TRY(ws.get(&m->col_bits, m->col_bits_words, true));
  return OCF_OK;
}

extern "C" int ocf_model_create(const ocf_model_config* cfg, ocf_model** out) {
  OCF_REQUIRE(cfg && out, "ocf_model_create: null argument");
  *out = nullptr;
  OCF_REQUIRE(cfg->n_cols > 0 && cfg->n_cols_total >= cfg->n_cols, "ocf_model_create: bad n_cols");
  OCF_REQUIRE(cfg->n_layers >= 1 && cfg->n_layers <= 8, "ocf_model_create: n_layers must be 1..8");
  OCF_REQUIRE(cfg->aux >= OCF_AUX_NONE && cfg->aux <= OCF_AUX_BOTH, "ocf_model_create: bad aux");
  OCF_REQUIRE(cfg->activation >= OCF_ACT_LINEAR && cfg->activation <= OCF_ACT_SOFTPLUS, "ocf_model_create: bad activation");
  OCF_REQUIRE(cfg->loss == OCF_LOSS_MSE || cfg->loss == OCF_LOSS_MAE, "ocf_model_create: bad loss");
  OCF_REQUIRE(cfg->max_rows > 0 && cfg->max_rows <= MAX_BATCH_ROWS, "ocf_model_create: max_rows must be 1..4096");
  OCF_REQUIRE(cfg->max_entries > 0 && cfg->max_entries < (int64_t(1) << 31), "ocf_model_create: bad max_entries");
  OCF_REQUIRE(cfg->dropout_p < 1.0f, "ocf_model_create: dropout_p must be < 1");
  for (int l = 0; l < cfg->n_layers; ++l)
    OCF_REQUIRE(cfg->widths[l] > 0 && cfg->widths[l] <= MAX_HP, "ocf_model_create: hidden widths must be 1..1024");
  ocf_model* m = new ocf_model();
  m->cfg = *cfg;
  m->L = cfg->n_layers;
  aux_bits(cfg->aux, m->nblk, m->bits);
  const int L = m->L, N = cfg->n_cols;
  for (int l = 0; l < L; ++l) m->hp.push_back(pad_h(cfg->widths[l]));
  m->layers.resize(L + 1);
  int st = OCF_OK;
  auto bail = [&](int code) { m->mem.release(); m->opt_mem.release(); m->ws_mem.release(); if (m->h_rec) cudaFreeHost(m->h_rec); delete m; return code; };
  for (int l = 0; l <= L && !st; ++l) {
    Layer& ly = m->layers[l];
    if (l == 0) { ly.fan_in = m->nblk * N; ly.fan_out = cfg->widths[0]; ly.rows = m->nblk * N; ly.hp = m->hp[0]; ly.bias_len = m->hp[0]; }
    else if (l < L) { ly.fan_in = cfg->widths[l - 1]; ly.fan_out = cfg->widths[l]; ly.rows = m->hp[l - 1]; ly.hp = m->hp[l]; ly.bias_len = m->hp[l]; }
    else { ly.fan_in = cfg->widths[L - 1]; ly.fan_out = N; ly.rows = N; ly.hp = m->hp[L - 1]; ly.bias_len = N; }
    // the decoder kernel is padded (zeros) to whole 256-column pair tiles of the scoring GEMM
    st = m->mem.get(&ly.W, (l == L ? align_up((size_t)ly.rows, 2 * tc::TILE_M) : (size_t)ly.rows) * ly.hp, true);
    if (!st) st = m->mem.get(&ly.b, (size_t)ly.bias_len, true);
  }
  if (st) return bail(st);
  if ((st = m->mem.get(&m->regparts, (size_t)N_REGPART * (L + 1), true)) || (st = m->mem.get(&m->d_step, 1, true)) ||
      (st = m->mem.get(&m->col_tasks, (size_t)N * (m->nblk + 1))) || (st = m->mem.get(&m->col_heavy, (size_t)N * (m->nblk + 1))) || (st = m->mem.get(&m->col_seg, (size_t)N, true)) ||
      (st = m->mem.get(&m->col_counters, 8, true)) || (st = m->mem.get(&m->col_state, (size_t)2 * N, true)) ||
      (st = m->mem.get(&m->col_info, (size_t)N)))
    return bail(st);
  { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&m->sm_count, cudaDevAttrMultiProcessorCount, dev); if (m->sm_count <= 0) m->sm_count = 148; }
  if ((st = alloc_workspace(m, cfg->max_rows, cfg->max_entries))) return bail(st);
  if (cudaHostAlloc(reinterpret_cast<void**>(&m->h_rec), sizeof(float) * LOG_CAP * LOG_W, cudaHostAllocMapped) != cudaSuccess ||
      cudaHostGetDevicePointer(reinterpret_cast<void**>(&m->h_rec_dev), m->h_rec, 0) != cudaSuccess)
    return bail(fail(OCF_ERR_NOMEM, "ocf_model_create: pinned allocation failed"));
  std::memset(m->h_rec, 0, sizeof(float) * LOG_CAP * LOG_W);
  for (int k = 0; k < 64; ++k)
    if (cudaEventCreateWithFlags(&m->step_ev[k], cudaEventDisableTiming) != cudaSuccess)
      return bail(fail(OCF_ERR_CUDA, "ocf_model_create: event creation failed"));
  // the column grouping (K4a) runs beside K2/K3 at the LOWEST priority: its small latency-bound CTAs take the
  // slots the row-centric kernels leave, instead of pushing those into a second wave; the capture stream carries
  // the highest priority so that captured steps keep the same order of preference
  int prio_lo = 0, prio_hi = 0;
  cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
  if (cudaStreamCreateWithPriority(&m->side, cudaStreamNonBlocking, prio_lo) != cudaSuccess ||
      cudaStreamCreateWithPriority(&m->cap, cudaStreamNonBlocking, prio_hi) != cudaSuccess ||
      cudaEventCreateWithFlags(&m->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&m->ev_join, cudaEventDisableTiming) != cudaSuccess ||
      cudaStreamCreateWithPriority(&m->side2, cudaStreamNonBlocking, prio_hi) != cudaSuccess ||
      cudaEventCreateWithFlags(&m->ev_fork2, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&m->ev_join2, cudaEventDisableTiming) != cudaSuccess)
    return bail(fail(OCF_ERR_CUDA, "ocf_model_create: side stream creation failed"));
  for (int k = 0; k < 8; ++k)
    if (cudaEventCreateWithFlags(&m->ev_dz[k], cudaEventDisableTiming) != cudaSuccess)
      return bail(fail(OCF_ERR_CUDA, "ocf_model_create: event creation failed"));
  *out = m;
  st = ocf_model_set_optimizer(m, OCF_OPT_ADAGRAD, 0.005f, 0.9f, 0.999f, 1e-8f, 0.f);   // train.py:50-51
  if (st) { *out = nullptr; return bail(st); }
  return OCF_OK;
}

extern "C" int ocf_model_destroy(ocf_model* m) {
  if (m) {
    cudaDeviceSynchronize();
    m->mem.release(); m->opt_mem.release(); m->dense_mem.release(); m->ws_mem.release(); m->par_mem.release();
    if (m->h_rec) cudaFreeHost(m->h_rec);
    for (int k = 0; k < 64; ++k) if (m->step_ev[k]) cudaEventDestroy(m->step_ev[k]);
    drop_graphs(m);
    if (m->side) cudaStreamDestroy(m->side);
    if (m->cap) cudaStreamDestroy(m->cap);
    if (m->ev_fork) cudaEventDestroy(m->ev_fork);
    if (m->ev_join) cudaEventDestroy(m->ev_join);
    if (m->side2) cudaStreamDestroy(m->side2);
    if (m->ev_fork2) cudaEventDestroy(m->ev_fork2);
    if (m->ev_join2) cudaEventDestroy(m->ev_join2);
    for (int k = 0; k < 8; ++k) if (m->ev_dz[k]) cudaEventDestroy(m->ev_dz[k]);
    delete m;
  }
  return OCF_OK;
}

extern "C" int ocf_model_reserve(ocf_model* m, int32_t max_rows, int64_t max_entries) {
  OCF_REQUIRE(m, "ocf_model_reserve: null argument");
  OCF_REQUIRE(max_rows > 0 && max_rows <= MAX_BATCH_ROWS && max_entries > 0 && max_entries < (int64_t(1) << 31), "ocf_model_reserve: bad sizes");
  if (max_rows <= m->cfg.max_rows && max_entries <= m->cfg.max_entries) return OCF_OK;
  OCF_CUDA(cudaDeviceSynchronize());
  return alloc_workspace(m, std::max(max_rows, m->cfg.max_rows), std::max(max_entries, m->cfg.max_entries));
}

extern "C" int ocf_model_num_weights(const ocf_model* m) { return m ? 2 * (m->L + 1) : 0; }

extern "C" int ocf_model_weight_shape(const ocf_model* m, int index, int64_t shape[2]) {
  OCF_REQUIRE(m && shape && index >= 0 && index < 2 * (m->L + 1), "ocf_model_weight_shape: bad argument");
  const Layer& ly = m->layers[index / 2];
  if (index % 2 == 0) { shape[0] = ly.fan_in; shape[1] = ly.fan_out; }
  else { shape[0] = ly.fan_out; shape[1] = 1; }
  return OCF_OK;
}

// Keras layout <-> internal layout. Kernels of layers 0..L-1: [fan_in, fan_out] -> [rows, hp]
// (fan_out padded); decoder kernel [H, N] -> transposed [N, hp].
static int weight_io(const ocf_model* m, int index, float* host, int64_t count, bool to_device) {
  const int l = index / 2;
  const Layer& ly = m->layers[l];
  const bool is_bias = index % 2 == 1;
  const bool dec = l == m->L;
  if (is_bias) {
    OCF_REQUIRE(count == ly.fan_out, "weight i/o: wrong element count");
    if (to_device) OCF_CUDA(cudaMemcpy(ly.b, host, sizeof(float) * ly.fan_out, cudaMemcpyHostToDevice));
    else OCF_CUDA(cudaMemcpy(host, ly.b, sizeof(float) * ly.fan_out, cudaMemcpyDeviceToHost));
    return OCF_OK;
  }
  OCF_REQUIRE(count == (int64_t)ly.fan_in * ly.fan_out, "weight i/o: wrong element count");
  if (!dec) {
    const size_t spitch = sizeof(float) * ly.fan_out, dpitch = sizeof(float) * ly.hp;
    if (to_device) OCF_CUDA(cudaMemcpy2D(ly.W, dpitch, host, spitch, spitch, ly.fan_in, cudaMemcpyHostToDevice));
    else OCF_CUDA(cudaMemcpy2D(host, spitch, ly.W, dpitch, spitch, ly.fan_in, cudaMemcpyDeviceToHost));
    return OCF_OK;
  }
  // decoder: transpose through a host block of <= 32768 catalogue columns at a time
  const int H = ly.fan_in, N = ly.fan_out, hp = ly.hp;
  const int blk = 32768;
  std::vector<float> tmp((size_t)std::min(blk, N) * hp);
  for (int c0 = 0; c0 < N; c0 += blk) {
    const int nc = std::min(blk, N - c0);
    if (to_device) {
      std::fill(tmp.begin(), tmp.end(), 0.f);
      for (int k = 0; k < H; ++k) {
        const float* src = host + (size_t)k * N + c0;
        for (int c = 0; c < nc; ++c) tmp[(size_t)c * hp + k] = src[c];
      }
      OCF_CUDA(cudaMemcpy(ly.W + (size_t)c0 * hp, tmp.data(), sizeof(float) * (size_t)nc * hp, cudaMemcpyHostToDevice));
    } else {
      OCF_CUDA(cudaMemcpy(tmp.data(), ly.W + (size_t)c0 * hp, sizeof(float) * (size_t)nc * hp, cudaMemcpyDeviceToHost));
      for (int k = 0; k < H; ++k) {
        float* dst = host + (size_t)k * N + c0;
        for (int c = 0; c < nc; ++c) dst[c] = tmp[(size_t)c * hp + k];
      }
    }
  }
  return OCF_OK;
}

extern "C" int ocf_model_set_weight(ocf_model* m, int index, const float* host, int64_t count) {
  OCF_REQUIRE(m && host && index >= 0 && index < 2 * (m->L + 1), "ocf_model_set_weight: bad argument");
  OCF_CUDA(cudaDeviceSynchronize());
  return weight_io(m, index, const_cast<float*>(host), count, true);
}

extern "C" int ocf_model_get_weight(const ocf_model* m, int index, float* host, int64_t count) {
  OCF_REQUIRE(m && host && index >= 0 && index < 2 * (m->L + 1), "ocf_model_get_weight: bad argument");
  OCF_CUDA(cudaDeviceSynchronize());
  return weight_io(m, index, host, count, false);
}

extern "C" int ocf_model_reset_optimizer(ocf_model* m) {
  OCF_REQUIRE(m, "ocf_model_reset_optimizer: null argument");
  OCF_CUDA(cudaDeviceSynchronize());
  m->iterations = 0;
  for (Layer& ly : m->layers) {
    if (ly.Ws1) OCF_CUDA(cudaMemset(ly.Ws1, 0, sizeof(float) * (size_t)ly.rows * ly.hp));
    if (ly.Ws2) OCF_CUDA(cudaMemset(ly.Ws2, 0, sizeof(float) * (size_t)ly.rows * ly.hp));
    if (ly.bs1) OCF_CUDA(cudaMemset(ly.bs1, 0, sizeof(float) * ly.bias_len));
    if (ly.bs2) OCF_CUDA(cudaMemset(ly.bs2, 0, sizeof(float) * ly.bias_len));
  }
  return OCF_OK;
}

extern "C" int ocf_model_set_optimizer(ocf_model* m, int kind, float lr, float p1, float p2, float epsilon, float decay) {
  OCF_REQUIRE(m, "ocf_model_set_optimizer: null argument");
  OCF_REQUIRE(kind >= OCF_OPT_SGD && kind <= OCF_OPT_ADAM, "ocf_model_set_optimizer: bad kind");
  OCF_CUDA(cudaDeviceSynchronize());
  drop_graphs(m);
  m->step_mirror_valid = false;
  const bool s1 = kind != OCF_OPT_SGD, s2 = kind == OCF_OPT_ADAM;
  if (s1 != m->has_s1 || s2 != m->has_s2) {
    m->opt_mem.release();
    for (Layer& ly : m->layers) { ly.Ws1 = ly.Ws2 = ly.bs1 = ly.bs2 = nullptr; }
    for (Layer& ly : m->layers) {
      if (s1) { OCF_TRY(m->opt_mem.get(&ly.Ws1, (size_t)ly.rows * ly.hp, true)); OCF_TRY(m->opt_mem.get(&ly.bs1, (size_t)ly.bias_len, true)); }
      if (s2) { OCF_TRY(m->opt_mem.get(&ly.Ws2, (size_t)ly.rows * ly.hp, true)); OCF_TRY(m->opt_mem.get(&ly.bs2, (size_t)ly.bias_len, true)); }
    }
    m->has_s1 = s1; m->has_s2 = s2;
  }
  m->opt_kind = kind; m->lr = lr; m->p1 = p1; m->p2 = p2; m->eps = epsilon; m->decay = decay;
  return ocf_model_reset_optimizer(m);
}

extern "C" int ocf_model_set_loss(ocf_model* m, int loss, float rating_range) {
  OCF_REQUIRE(m && (loss == OCF_LOSS_MSE || loss == OCF_LOSS_MAE), "ocf_model_set_loss: bad argument");
  if (m->cfg.loss != loss || m->cfg.rating_range != rating_range) drop_graphs(m);
  m->cfg.loss = loss;
  m->cfg.rating_range = rating_range;
  return OCF_OK;
}

extern "C" int ocf_model_set_aux(ocf_model* m, int aux) {
  OCF_REQUIRE(m && aux >= OCF_AUX_NONE && aux <= OCF_AUX_BOTH, "ocf_model_set_aux: bad argument");
  int nblk; int3 bits;
  aux_bits(aux, nblk, bits);
  OCF_REQUIRE(nblk == m->nblk, "ocf_model_set_aux: this mask type feeds a different number of input blocks than the model has");
  if (m->cfg.aux != aux) drop_graphs(m);
  m->cfg.aux = aux; m->bits = bits;
  return OCF_OK;
}

extern "C" int ocf_model_set_trainable(ocf_model* m, int layer, int trainable) {
  OCF_REQUIRE(m && layer >= 0 && layer <= m->L, "ocf_model_set_trainable: bad argument");
  if (m->layers[layer].trainable != (trainable != 0)) drop_graphs(m);
  m->layers[layer].trainable = trainable != 0;
  return OCF_OK;
}

extern "C" int64_t ocf_model_steps_logged(const ocf_model* m) { return m ? m->steps_logged : 0; }

extern "C" int ocf_model_buffer(ocf_model* m, int which, void** ptr, int64_t* count) {
  OCF_REQUIRE(m && ptr && count, "ocf_model_buffer: null argument");
  switch (which) {
    case OCF_BUF_Z: *ptr = m->zsum[0]; *count = (int64_t)m->cfg.max_rows * m->hp[0]; break;
    case OCF_BUF_DH: *ptr = m->dh_top; *count = (int64_t)m->cfg.max_rows * m->hp[m->L - 1]; break;
    case OCF_BUF_ROWSTATS: *ptr = m->rowstats; *count = (int64_t)m->cfg.max_rows * ROWSTAT_W; break;
    case OCF_BUF_STATS_DH: *ptr = m->rowstats; *count = (int64_t)m->cfg.max_rows * (ROWSTAT_W + m->hp[m->L - 1]); break;
    default: return fail(OCF_ERR_INVALID, "ocf_model_buffer: unknown buffer");
  }
  return OCF_OK;
}

extern "C" int ocf_model_weight_device(ocf_model* m, int index, void** ptr, int64_t* count) {
  OCF_REQUIRE(m && ptr && count && index >= 0 && index < 2 * (m->L + 1), "ocf_model_weight_device: bad argument");
  const Layer& ly = m->layers[index / 2];
  if (index % 2 == 0) { *ptr = ly.W; *count = (int64_t)ly.rows * ly.hp; }
  else { *ptr = ly.b; *count = ly.bias_len; }
  return OCF_OK;
}

// ============================================================================================
// step orchestration
// ============================================================================================
#define OCF_NV_SWITCH(hp, ...)                                   \
  switch ((hp) / 128) {                                          \
    case 1: { constexpr int NV = 1; __VA_ARGS__; } break;        \
    case 2: { constexpr int NV = 2; __VA_ARGS__; } break;        \
    case 3: { constexpr int NV = 3; __VA_ARGS__; } break;        \
    case 4: { constexpr int NV = 4; __VA_ARGS__; } break;        \
    case 5: { constexpr int NV = 5; __VA_ARGS__; } break;        \
    case 6: { constexpr int NV = 6; __VA_ARGS__; } break;        \
    case 7: { constexpr int NV = 7; __VA_ARGS__; } break;        \
    default: { constexpr int NV = 8; __VA_ARGS__; } break;       \
  }

static OptDev make_opt(const ocf_model* m) {
  OptDev o{};
  o.kind = m->opt_kind;
  double lr = (double)m->lr;
  if (m->decay > 0.f) lr *= 1.0 / (1.0 + (double)m->decay * (double)m->iterations);
  if (m->opt_kind == OCF_OPT_ADAM) {
    const double t = (double)(m->iterations + 1);
    lr *= std::sqrt(1.0 - std::pow((double)m->p2, t)) / (1.0 - std::pow((double)m->p1, t));
  }
  o.lr = (float)lr;
  o.p1 = m->p1; o.one_m_p1 = (float)(1.0 - (double)m->p1);
  o.p2 = m->p2; o.one_m_p2 = (float)(1.0 - (double)m->p2);
  o.eps = m->eps;
  o.l2x2 = m->cfg.l2 >= 0.f ? (float)(2.0 * (double)m->cfg.l2) : 0.f;
  o.dense = (m->opt_kind == OCF_OPT_RMSPROP || m->opt_kind == OCF_OPT_ADAM || o.l2x2 != 0.f) ? 1 : 0;
  o.st = m->d_step;                 // the kernels read this step's lr there (sync_step_state keeps it current)
  return o;
}

static int check_step(const ocf_model* m, const ocf_batch* b, bool train) {
  OCF_REQUIRE(m && b, "step: null argument");
  if (b->mode == 0) return fail(OCF_ERR_STATE, "step: the batch has not been filled");
  if (train && b->mode != 1) return fail(OCF_ERR_STATE, "train step needs a split batch (ocf_batch_fill_split)");
  OCF_REQUIRE(b->store->n_cols == m->cfg.n_cols, "step: the batch's store and the model disagree on n_cols");
  OCF_REQUIRE(b->dev.B <= m->cfg.max_rows && b->dev.n_entries <= m->cfg.max_entries && b->dev.n_items <= m->max_items,
              "step: the batch exceeds the model's workspace");
  return OCF_OK;
}

// Makes the device-resident step scalars what this step needs: the caller's dropout counter / seed,
// the host's log slot and this step's learning rate. The kernels advance step and log_slot themselves,
// so a plain training loop never rewrites them (Adam and `decay` change lr every step and do).
static int sync_step_state(ocf_model* m, const ocf_step_args* args, cudaStream_t st) {
  StepDev want{};
  want.step = args ? args->step : 0u;
  want.log_slot = (int32_t)(m->steps_logged % LOG_CAP);
  want.lr = make_opt(m).lr;
  const uint64_t seed = args ? args->dropout_seed : 0;
  want.seed_lo = (uint32_t)(seed & 0xffffffffu); want.seed_hi = (uint32_t)(seed >> 32);
  const StepDev& have = m->step_mirror;
  if (m->step_mirror_valid && have.step == want.step && have.log_slot == want.log_slot && have.lr == want.lr &&
      have.seed_lo == want.seed_lo && have.seed_hi == want.seed_hi)
    return OCF_OK;
  k_set_step<<<1, 1, 0, st>>>(m->d_step, want);
  OCF_LAUNCHED();
  m->step_mirror = want;
  m->step_mirror_valid = true;
  return OCF_OK;
}

// Work-item grids: a captured step must cover any later fill of the same batch object, so it
// launches the batch's item capacity (CTAs beyond the header's n_items return at once).
static inline int item_grid(const ocf_model* m, const ocf_batch* b) {
  return m->capturing ? std::min(b->max_items, m->max_items) : b->dev.n_items;
}

static ActArgs act_args(ocf_model* m, int l, int B, bool training, const ocf_step_args* args) {
  const int hp = m->hp[l];
  const bool drop = training && m->cfg.dropout_p > 0.f;
  ActArgs g{};
  g.bias = reinterpret_cast<const float4*>(m->layers[l].b); g.B = B; g.H = m->cfg.widths[l]; g.hp4 = hp / 4;
  g.act = m->cfg.activation;
  g.a_out = reinterpret_cast<float4*>(m->act[l]);
  g.h_out = reinterpret_cast<float4*>(drop ? m->h[l] : m->act[l]);
  g.dscale = drop ? reinterpret_cast<float4*>(m->dscale[l]) : nullptr;
  g.p_drop = m->cfg.dropout_p;
  g.st = m->d_step; g.layer = (uint32_t)l; g.row0 = args ? args->row0 : 0;
  return g;
}

// phase 1: encoder partial sums; the row tails leave either z (z_out, or zsum[0]) or, with `fuse_act`,
// the first layer's activations (bias + activation + dropout applied by the row's last CTA).
static int phase_encode(ocf_model* m, const ocf_batch* b, cudaStream_t st, float* z_out, bool fuse_act, bool training,
                        const ocf_step_args* args) {
  const BatchDev& bt = b->dev;
  const int hp0 = m->hp[0];
  const ActArgs act = act_args(m, 0, bt.B, training, args);
  float4* z = reinterpret_cast<float4*>(z_out ? z_out : m->zsum[0]);
  g_prof.begin(1, st);
  OCF_NV_SWITCH(hp0, k_enc_fwd<NV><<<item_grid(m, b), 128, 0, st>>>(bt, m->layers[0].W, m->cfg.n_cols, m->nblk, m->bits,
                                                                     reinterpret_cast<float4*>(m->P1), m->tail, z, fuse_act ? 1 : 0, act));
  OCF_LAUNCHED();
  g_prof.end(1, st);
  return OCF_OK;
}

// bias + activation (+ dropout) of layer l from zsum[l]
static int launch_act(ocf_model* m, int l, int B, bool training, const ocf_step_args* args, cudaStream_t st) {
  const int hp = m->hp[l];
  const int total = B * (hp / 4);
  k_bias_act<<<(total + 255) / 256, 256, 0, st>>>(reinterpret_cast<const float4*>(m->zsum[l]), act_args(m, l, B, training, args));
  OCF_LAUNCHED();
  return OCF_OK;
}

// ---- hidden [H1, H2] layers on the tensor cores (ocf_gemm_tc.cuh) ----
// a_l = act(h_{l-1} . W_l + b_l) (+ dropout): D[n, b] = sum_k W[k, n] h[b, k]
static int hidden_fwd_tc(ocf_model* m, int l, int B, const float* hin, const ActArgs& act, cudaStream_t st, bool pdl = false) {
  CUtensorMap ma, mb;
  OCF_TRY(gtc::make_map_mn(&ma, m->layers[l].W, m->hp[l], m->hp[l], m->hp[l - 1]));
  OCF_TRY(gtc::make_map_k(&mb, hin, m->hp[l - 1], m->hp[l - 1], B));
  gtc::GemmTcArgs g{};
  g.kind = gtc::GEPI_FWD; g.a_mn = 1; g.b_mn = 0; g.actargs = act;
  g_prof.begin(8, st);
  OCF_TRY(gtc::launch(ma, mb, g, m->hp[l], B, m->hp[l - 1], st, 0, pdl && !g_prof.on));
  g_prof.end(8, st);
  return OCF_OK;
}

// dz_{l-1} = (dz_l . W_l^T) * dropout scale * act'(a_{l-1}): D[k, b] = sum_n W[k, n] dz[b, n]
static int hidden_dz_tc(ocf_model* m, int l, int B, bool drop, cudaStream_t st, bool pdl = false) {
  CUtensorMap ma, mb;
  OCF_TRY(gtc::make_map_k(&ma, m->layers[l].W, m->hp[l], m->hp[l], m->hp[l - 1]));
  OCF_TRY(gtc::make_map_k(&mb, m->dz[l], m->hp[l], m->hp[l], B));
  gtc::GemmTcArgs g{};
  g.kind = gtc::GEPI_DZ; g.a_mn = 0; g.b_mn = 0;
  g.C = m->dz[l - 1]; g.ldc = m->hp[l - 1]; g.aux0 = m->act[l - 1]; g.aux1 = drop ? m->dscale[l - 1] : nullptr; g.act = m->cfg.activation;
  g_prof.begin(8, st);
  OCF_TRY(gtc::launch(ma, mb, g, m->hp[l - 1], B, m->hp[l], st, 0, pdl && !g_prof.on));
  g_prof.end(8, st);
  return OCF_OK;
}

// dW_l = h_{l-1}^T . dz_l fused with the update of W_l (or stored, row-parallel mode): D[n, k] = sum_b dz[b, n] h[b, k]
static int hidden_dw_tc(ocf_model* m, int l, int B, const float* hin, const OptDev& opt, float* grad_out, cudaStream_t st, bool pdl = false) {
  Layer& ly = m->layers[l];
  CUtensorMap ma, mb;
  OCF_TRY(gtc::make_map_mn(&ma, m->dz[l], m->hp[l], m->hp[l], B));
  OCF_TRY(gtc::make_map_mn(&mb, hin, m->hp[l - 1], m->hp[l - 1], B));
  gtc::GemmTcArgs g{};
  g.a_mn = 1; g.b_mn = 1; g.ldc = m->hp[l];
  if (grad_out) { g.kind = gtc::GEPI_STORE; g.C = grad_out; }
  else { g.kind = gtc::GEPI_UPDATE; g.C = ly.W; g.s1 = ly.Ws1; g.s2 = ly.Ws2; g.opt = opt; }
  g_prof.begin(8, st);
  OCF_TRY(gtc::launch(ma, mb, g, m->hp[l], m->hp[l - 1], B, st, 0, pdl && !g_prof.on));
  g_prof.end(8, st);
  return OCF_OK;
}

// phase 2: activations, hidden layers, decoder at the target entries, loss partials -> dh_top, rowstats
// act0_done: the first layer's activations are already in place (fused into the encoder's row tails or
// into the exchange).
// after_kernel: the previous operation in the stream is a kernel (the phase's first launch may be a dependent launch)
// An unsharded model's K3 leaves dz of the top hidden layer itself (DzFuse): dL/dh of a row is complete on this device.
// A column shard all-reduces dL/dh first and keeps the separate kernel.
static bool fuse_dz(const ocf_model* m) { return !m->cfg.sharded && m->par_mode == 0; }

static int phase_decode(ocf_model* m, const ocf_batch* b, bool training, const ocf_step_args* args,
                        float* dense_out, cudaStream_t st, bool act0_done = false, bool after_kernel = false) {
  const BatchDev& bt = b->dev;
  const int L = m->L, B = bt.B;
  const bool drop = training && m->cfg.dropout_p > 0.f;
  bool dep = after_kernel && !g_prof.on;       // instrumented passes record events between the kernels
  if (!act0_done) { OCF_TRY(launch_act(m, 0, B, training, args, st)); dep = !g_prof.on; }
  for (int l = 1; l < L; ++l) {
    // hidden layer: product + bias + activation + dropout in the GEMM's epilogue
    const float* hin = drop ? m->h[l - 1] : m->act[l - 1];
    OCF_TRY(hidden_fwd_tc(m, l, B, hin, act_args(m, l, B, training, args), st, dep));
    dep = !g_prof.on;
  }
  const float* htop = drop ? m->h[L - 1] : m->act[L - 1];
  const int hpt = m->hp[L - 1];
  const int rows_total = (args && args->rows_total > 0) ? args->rows_total : B;
  const double bn = (double)rows_total * (double)m->cfg.n_cols_total;
  const float gscale = (float)((m->cfg.loss == OCF_LOSS_MSE ? 2.0 : 1.0) / bn);
  float* stats_out = m->rowstats;
  float4* dh_out = reinterpret_cast<float4*>(m->dh_top);
  DzFuse fz{};
  if (training && fuse_dz(m)) {
    fz.a = reinterpret_cast<const float4*>(m->act[L - 1]);
    fz.dscale = drop ? reinterpret_cast<const float4*>(m->dscale[L - 1]) : nullptr;
    fz.dz = reinterpret_cast<float4*>(m->dz[L - 1]);
    fz.act = m->cfg.activation;
  }
  g_prof.begin(2, st);
  if (training) {
    OCF_NV_SWITCH(hpt, OCF_CUDA(launch_pdl(dep, k_dec_fwd<NV, true>, dim3(item_grid(m, b)), dim3(128), st, bt, (const float*)m->layers[L].W,
                                           (const float*)m->layers[L].b, htop, gscale, m->cfg.loss, m->dy, reinterpret_cast<float4*>(m->P2),
                                           m->itemstats, dense_out, m->cfg.n_cols, m->tail, dh_out, stats_out, fz)));
  } else {
    OCF_NV_SWITCH(hpt, OCF_CUDA(launch_pdl(dep, k_dec_fwd<NV, false>, dim3(item_grid(m, b)), dim3(128), st, bt, (const float*)m->layers[L].W,
                                           (const float*)m->layers[L].b, htop, gscale, m->cfg.loss, (float*)nullptr, (float4*)nullptr,
                                           m->itemstats, dense_out, m->cfg.n_cols, m->tail, (float4*)nullptr, stats_out, fz)));
  }
  OCF_LAUNCHED();
  g_prof.end(2, st);
  return OCF_OK;
}

static MetricArgs metric_args(ocf_model* m, int B, const ocf_step_args* args, int n_reg, bool advance_step, const float* stats = nullptr) {
  const int rows_total = (args && args->rows_total > 0) ? args->rows_total : B;
  MetricArgs a{};
  a.rowstats = stats ? stats : m->rowstats; a.rows = B; a.rows_total = (float)rows_total;
  a.n_cols_total = (float)m->cfg.n_cols_total; a.rating_range = m->cfg.rating_range; a.loss_kind = m->cfg.loss;
  a.regparts = m->regparts; a.n_reg = n_reg; a.l2 = m->cfg.l2 >= 0.f ? m->cfg.l2 : 0.f;
  a.log = m->h_rec_dev; a.st = m->d_step; a.advance_step = advance_step ? 1 : 0;
  return a;
}

// A step's record is written into page-locked host memory by its own kernel; readers wait on the step's
// event instead of the whole stream. Also advances the host's mirror of the device-side step scalars.
static int publish_metrics(ocf_model* m, bool trained, cudaStream_t st) {
  OCF_CUDA(cudaEventRecord(m->step_ev[m->steps_logged % 64], st));
  m->steps_logged += 1;
  m->step_mirror.log_slot = (int32_t)(m->steps_logged % LOG_CAP);
  if (trained) m->step_mirror.step += 1u;
  return OCF_OK;
}

static int launch_metrics(ocf_model* m, int B, const ocf_step_args* args, int n_reg, bool trained, cudaStream_t st,
                          const float* stats = nullptr) {
  k_metrics<<<1, 32, 0, st>>>(metric_args(m, B, args, n_reg, trained, stats));
  OCF_LAUNCHED();
  return OCF_OK;
}

static int launch_reg(ocf_model* m, cudaStream_t st) {
  if (m->cfg.l2 < 0.f) return 0;
  for (int l = 0; l <= m->L; ++l) {
    const Layer& ly = m->layers[l];
    k_sumsq<<<N_REGPART, 256, 0, st>>>(ly.W, (size_t)ly.rows * ly.hp, m->regparts + (size_t)l * N_REGPART);
    g_launches.fetch_add(1);
  }
  return N_REGPART * (m->L + 1);
}

template <int NV, bool WIDE, bool HEAVY>
static int launch_row_update_nv(int kind, int grid, const RowArgs& r, cudaStream_t st, bool dep) {
  const dim3 g(grid), b(256);
  switch (kind) {
    case OCF_OPT_SGD: OCF_CUDA(launch_pdl(dep, k_row_update<NV, OCF_OPT_SGD, WIDE, HEAVY>, g, b, st, r)); break;
    case OCF_OPT_ADAGRAD: OCF_CUDA(launch_pdl(dep, k_row_update<NV, OCF_OPT_ADAGRAD, WIDE, HEAVY>, g, b, st, r)); break;
    case OCF_OPT_RMSPROP: OCF_CUDA(launch_pdl(dep, k_row_update<NV, OCF_OPT_RMSPROP, WIDE, HEAVY>, g, b, st, r)); break;
    case KIND_GRAD: OCF_CUDA(launch_pdl(dep, k_row_update<NV, KIND_GRAD, false, false>, g, b, st, r)); break;
    default: OCF_CUDA(launch_pdl(dep, k_row_update<NV, OCF_OPT_ADAM, WIDE, HEAVY>, g, b, st, r)); break;
  }
  OCF_LAUNCHED();
  return OCF_OK;
}

static int launch_row_update(int hp, int kind, int sm_count, bool wide, bool heavy, const RowArgs& r, cudaStream_t st, bool dep) {
  const int grid = sm_count * (wide ? 4 : 6);
  if (wide) { OCF_NV_SWITCH(hp, return (launch_row_update_nv<NV, true, true>(kind, grid, r, st, dep))); }
  else if (heavy) { OCF_NV_SWITCH(hp, return (launch_row_update_nv<NV, false, true>(kind, grid, r, st, dep))); }
  else { OCF_NV_SWITCH(hp, return (launch_row_update_nv<NV, false, false>(kind, grid, r, st, dep))); }
  return OCF_OK;
}

// Catalogues whose weights are within reach of the 126 MB L2 (n_cols x hp <= 32 M floats): the update is bound by its
// longest chain of dependent L2 round trips, so long chains are split over a CTA; beyond that it is HBM-bound.
static bool heavy_model(const ocf_model* m) {
  return (size_t)m->cfg.n_cols * (size_t)std::max(m->hp[0], m->hp[m->L - 1]) <= ((size_t)32 << 20);
}

// The model's own work list (filled inside the step).
static WorkList model_wl(const ocf_model* m) {
  WorkList w;
  w.matches = m->col_matches; w.entries = m->cfg.max_entries; w.seg = m->col_seg; w.tasks = m->col_tasks; w.heavy = m->col_heavy;
  w.counters = m->col_counters; w.state = m->col_state; w.info = m->col_info; w.bits = m->col_bits;
  return w;
}

static WorkSig work_sig(const ocf_model* m, const ocf_batch* b) {
  WorkSig s;
  s.n_cols = m->cfg.n_cols; s.nblk = m->nblk; s.b0 = m->bits.x; s.b1 = m->bits.y; s.b2 = m->bits.z;
  s.do_dec = m->layers[m->L].trainable ? 1 : 0; s.do_enc = m->layers[0].trainable ? 1 : 0;
  s.dense = make_opt(m).dense; s.heavy = heavy_model(m) ? 1 : 0; s.B = b->dev.B; s.dups = b->store->has_dups ? 1 : 0;
  return s;
}
// The batch carries the work list of its current fill, built for this model's settings.
static bool wl_current(const ocf_model* m, const ocf_batch* b) {
  return m->par_mode == 0 && b->wl_seq != 0 && b->wl_seq == b->fill_seq && b->wl_sig == work_sig(m, b);
}
// The list this step's update walks.
static WorkList step_wl(const ocf_model* m, const ocf_batch* b) { return wl_current(m, b) ? b->wl : model_wl(m); }

// K4a: the batch's ratings grouped by catalogue column -> match list + update tasks.
// zeroed: the caller has already cleared the list's counters / per-column state (one memset over the batch's own list).
static int launch_scan(ocf_model* m, const ocf_batch* b, int do_dec, int do_enc, int dense, cudaStream_t st, const WorkList& wl,
                       bool zeroed = false) {
  if (!do_dec && !do_enc) return OCF_OK;
  const BatchDev& bt = b->dev;
  if (!zeroed) {
    OCF_CUDA(cudaMemsetAsync(wl.counters, 0, 8 * sizeof(int), st));
    if (dense) OCF_CUDA(cudaMemsetAsync(wl.seg, 0, sizeof(int2) * (size_t)m->cfg.n_cols, st));
  }
  const int dups = b->store->has_dups ? 1 : 0;
  const int W = (bt.B + 31) / 32;
  const size_t N = (size_t)m->cfg.n_cols;
  if (!zeroed) {
    OCF_CUDA(cudaMemsetAsync(wl.state, 0, sizeof(int) * 2 * N, st));
    OCF_CUDA(cudaMemsetAsync(wl.bits, 0, sizeof(uint32_t) * N * W, st));
  }
  // a row that repeats a column merges its ratings into one record per (column, batch row): fields without a
  // writer must read 0 (the whole capacity: a captured list graph serves every fill of the batch object)
  if (dups) OCF_CUDA(cudaMemsetAsync(wl.matches, 0, sizeof(uint32_t) * 3 * (size_t)wl.entries, st));
  SortArgs a{};
  a.bt = bt;
  a.cnt = wl.state; a.codeor = wl.state + N;
  a.colinfo = wl.info; a.bits = wl.bits; a.W = W; a.counters = wl.counters;
  a.matches = wl.matches; a.tasks = wl.tasks; a.colseg = wl.seg; a.heavy = heavy_model(m) ? wl.heavy : nullptr;
  a.n_cols = m->cfg.n_cols; a.nblk = m->nblk; a.bits3 = m->bits; a.dense = dense; a.do_dec = do_dec; a.do_enc = do_enc;
  a.dups = dups;
  const int grid = item_grid(m, b);
  g_prof.begin(3, st);
  k_sort_count<<<grid, 128, 0, st>>>(a);
  OCF_LAUNCHED();
  OCF_CUDA(launch_pdl(!g_prof.on, k_sort_alloc, dim3((m->cfg.n_cols + 255) / 256), dim3(256), st, a));
  OCF_LAUNCHED();
  OCF_CUDA(launch_pdl(!g_prof.on, k_sort_place, dim3(grid), dim3(128), st, a));
  OCF_LAUNCHED();
  g_prof.end(3, st);
  return OCF_OK;
}

// K4b: one warp per (column, array) task: gradient row from the matches, fused optimizer update.
static int launch_rows(ocf_model* m, const ocf_batch* b, int do_dec, int do_enc, int hpx, const OptDev& opt, cudaStream_t st,
                       bool grad_mode = false, int only = 0, bool after_kernel = true) {
  if (!do_dec && !do_enc) return OCF_OK;
  const int L = m->L;
  const bool drop = m->cfg.dropout_p > 0.f;
  Layer& enc = m->layers[0];
  Layer& dec = m->layers[L];
  RowArgs r{};
  const WorkList wl = step_wl(m, b);
  r.matches = wl.matches; r.tasks = wl.tasks; r.colseg = wl.seg; r.counters = wl.counters;
  // small catalogues (weights + state within reach of the 126 MB L2): latency-bound, wide walk; else HBM-bound
  const bool wide = !grad_mode && (size_t)m->cfg.n_cols * (size_t)hpx <= ((size_t)8 << 20);
  const bool heavy = heavy_model(m) && !grad_mode;      // exactly when K4a lists heavy tasks
  r.heavy = heavy ? wl.heavy : nullptr;
  r.hdec = drop ? m->h[L - 1] : m->act[L - 1]; r.dz0 = m->dz[0]; r.dy = m->dy;
  r.WdecT = dec.W; r.Wd_s1 = dec.Ws1; r.Wd_s2 = dec.Ws2; r.bdec = dec.b; r.bd_s1 = dec.bs1; r.bd_s2 = dec.bs2;
  r.Wenc = enc.W; r.We_s1 = enc.Ws1; r.We_s2 = enc.Ws2;
  r.n_cols = m->cfg.n_cols; r.bits = m->bits; r.bt_hdr = b->dev.hdr; r.opt = opt;
  r.task_cap = m->cfg.n_cols * (m->nblk + 1);
  r.dense = grad_mode ? 0 : opt.dense; r.n_arr = 0; r.only = only;
  if (grad_mode) { r.Gdec = m->gW[L]; r.Genc = m->gW[0]; r.gbdec = m->gb[L]; }
  if (do_dec) r.arr_map[r.n_arr++] = 0;
  if (do_enc) for (int blk = 0; blk < m->nblk; ++blk) r.arr_map[r.n_arr++] = 1 + blk;
  g_prof.begin(5, st);
  // a dependent launch: its predecessor in this stream is a kernel (the backward pass, or the first of two row updates)
  OCF_TRY(launch_row_update(hpx, grad_mode ? KIND_GRAD : opt.kind, m->sm_count, wide, heavy, r, st, after_kernel && !g_prof.on));
  g_prof.end(5, st);
  return OCF_OK;
}

// Start the column grouping of a training step on the side stream, ordered after everything already
// enqueued on `st` (the batch's gather, the previous step's update which reads the match list).
static int fork_scan(ocf_model* m, const ocf_batch* b, cudaStream_t st) {
  m->scan_pending = false;
  if (wl_current(m, b)) return OCF_OK;          // grouped ahead of the step on the batch's stream (prepare_worklist)
  const int L = m->L;
  const OptDev opt = make_opt(m);
  const int dense = m->par_mode == OCF_PAR_ROWS ? 0 : opt.dense;   // gradient rows exist for touched columns only
  const int do_dec = m->layers[L].trainable ? 1 : 0, do_enc = m->layers[0].trainable ? 1 : 0;
  if (!do_dec && !do_enc) return OCF_OK;
  OCF_CUDA(cudaEventRecord(m->ev_fork, st));
  OCF_CUDA(cudaStreamWaitEvent(m->side, m->ev_fork, 0));
  OCF_TRY(launch_scan(m, b, do_dec, do_enc, dense, m->side, model_wl(m)));
  OCF_CUDA(cudaEventRecord(m->ev_join, m->side));
  m->scan_pending = true;
  return OCF_OK;
}

// phase 3 (training): backward through the hidden layers, fused updates, metrics
// grad_mode (row-parallel): the same backward pass, but every gradient lands in the gradient arena
// (zeroed first: untouched weight rows have no gradient) and nothing is applied or logged; the
// caller all-reduces the arena and runs apply_gradients().
static int phase_update(ocf_model* m, const ocf_batch* b, const ocf_step_args* args, cudaStream_t st, bool grad_mode = false,
                        int* n_reg_out = nullptr, bool after_kernel = false) {
  const BatchDev& bt = b->dev;
  const int L = m->L, B = bt.B;
  const bool drop = m->cfg.dropout_p > 0.f;
  const OptDev opt = make_opt(m);
  const int n_reg = launch_reg(m, st);          // L2 term of the reported loss uses pre-update weights
  if (n_reg_out) *n_reg_out = n_reg;
  if (grad_mode) OCF_CUDA(cudaMemsetAsync(m->grads, 0, sizeof(float) * m->grads_count, st));
  Layer& enc = m->layers[0];
  Layer& dec = m->layers[L];
  const int hpd = m->hp[L - 1], hpe = m->hp[0];
  // What is not on the critical path K3 -> (backward products of the hidden layers) -> encoder rows runs on a second
  // stream beside it and joins at the end of the step:
  //   * the bias gradients (column sums of dz; K3 has already left dz of the top layer, fuse_dz) and, riding along
  //     with the first of them, the step's metric record;
  //   * the gradient product + update of hidden layer l: needs dz_l, and W_l no longer being read by the backward product;
  //   * the decoder rows' update: needs nothing after K3 (only when it is a real kernel: a catalogue of a few
  //     hundred columns updates in one small launch either way).
  const bool fz = fuse_dz(m) && !grad_mode;
  const bool side_ok = !grad_mode && m->par_mode == 0 && wl_current(m, b) && m->side2 != nullptr && !g_prof.on;
  const bool side_bias = side_ok && fz;
  const bool split_dw = side_ok && L > 1;
  const bool split = side_ok && L > 1 && (size_t)m->cfg.n_cols * (size_t)hpd >= ((size_t)1 << 20);
  bool forked = false;
  if (side_bias || (split && dec.trainable)) {
    OCF_CUDA(cudaEventRecord(m->ev_fork2, st));
    OCF_CUDA(cudaStreamWaitEvent(m->side2, m->ev_fork2, 0));
    forked = true;
  }
  // dependent launches (PDL) from here on whenever the previous operation in the stream is a kernel
  bool dep = (after_kernel || n_reg > 0) && !grad_mode && !g_prof.on;
  // top hidden layer: dz (unless K3 left it) and its bias
  {
    const int l = L - 1;
    Layer& ly = m->layers[l];
    // the fused step's metric record rides along as one extra CTA (a row-parallel step needs the
    // other ranks' row statistics first and computes it after the gather)
    MetricArgs met{};
    if (!grad_mode) met = metric_args(m, B, args, n_reg, true);
    OCF_CUDA(launch_pdl(side_bias ? false : dep, k_dz_bias, dim3(m->hp[l] / 32 + (grad_mode ? 0 : 1)), dim3(1024), side_bias ? m->side2 : st,
                        (const float*)(fz ? m->dz[l] : m->dh_top), (const float*)m->act[l],
                        (const float*)(drop ? m->dscale[l] : nullptr), B, m->hp[l], m->cfg.activation, fz ? 1 : 0, m->dz[l], ly.b, ly.bs1, ly.bs2, opt,
                        ly.trainable ? 1 : 0, grad_mode ? m->gb[l] : (float*)nullptr, met));
    OCF_LAUNCHED();
    if (!side_bias) dep = !g_prof.on;
  }
  if (split && dec.trainable) OCF_TRY(launch_rows(m, b, 1, 0, hpd, opt, m->side2, false, 1, side_bias));
  for (int l = L - 1; l >= 1; --l) {
    Layer& ly = m->layers[l];
    // dz_{l-1} = (dz_l . W_l^T) * dropout scale * act'(a_{l-1})   (uses W_l before its update)
    OCF_TRY(hidden_dz_tc(m, l, B, drop, st, dep));
    dep = !g_prof.on;
    const bool to_side = side_bias || (split_dw && ly.trainable);
    if (to_side) {
      OCF_CUDA(cudaEventRecord(m->ev_dz[l], st));
      OCF_CUDA(cudaStreamWaitEvent(m->side2, m->ev_dz[l], 0));
      forked = true;
    }
    Layer& lo = m->layers[l - 1];
    OCF_CUDA(launch_pdl(side_bias ? false : dep, k_dz_bias, dim3(m->hp[l - 1] / 32), dim3(1024), side_bias ? m->side2 : st, (const float*)m->dz[l - 1],
                        (const float*)nullptr, (const float*)nullptr,
                        B, m->hp[l - 1], m->cfg.activation, 1, m->dz[l - 1], lo.b, lo.bs1, lo.bs2, opt, lo.trainable ? 1 : 0,
                        grad_mode ? m->gb[l - 1] : (float*)nullptr, MetricArgs{}));
    OCF_LAUNCHED();
    if (ly.trainable) {
      // dW_l = h_{l-1}^T . dz_l, fused with the update of W_l
      const float* hin = drop ? m->h[l - 1] : m->act[l - 1];
      OCF_TRY(hidden_dw_tc(m, l, B, hin, opt, grad_mode ? m->gW[l] : nullptr, split_dw ? m->side2 : st, split_dw ? side_bias : dep));
    }
  }
  // catalogue-wide kernels: encoder rows and decoder rows of every touched column
  const int dense = grad_mode ? 0 : opt.dense;
  // decoder and encoder rows share one padded width in the reference's architectures (one
  // num_hidden_units). A width list with different ends shares the grouping too: its task list holds both kinds of
  // rows and each of the two launches (one per width) takes its own.
  if (wl_current(m, b)) {}                        // the batch brought its list along
  else if (m->scan_pending) { OCF_CUDA(cudaStreamWaitEvent(st, m->ev_join, 0)); m->scan_pending = false; }
  else OCF_TRY(launch_scan(m, b, dec.trainable ? 1 : 0, enc.trainable ? 1 : 0, dense, st, model_wl(m)));
  if (split) {
    OCF_TRY(launch_rows(m, b, 0, enc.trainable ? 1 : 0, hpe, opt, st, false, 2));       // the decoder rows are on their way
  } else if (hpd == hpe) {
    OCF_TRY(launch_rows(m, b, dec.trainable ? 1 : 0, enc.trainable ? 1 : 0, hpd, opt, st, grad_mode));
  } else {
    OCF_TRY(launch_rows(m, b, dec.trainable ? 1 : 0, 0, hpd, opt, st, grad_mode, 1));
    OCF_TRY(launch_rows(m, b, 0, enc.trainable ? 1 : 0, hpe, opt, st, grad_mode, 2));
  }
  if (forked) {
    OCF_CUDA(cudaEventRecord(m->ev_join2, m->side2));
    OCF_CUDA(cudaStreamWaitEvent(st, m->ev_join2, 0));
  }
  return OCF_OK;
}

extern "C" int ocf_model_wait_metrics(ocf_model* m, int64_t step, float* host) {
  OCF_REQUIRE(m && host, "ocf_model_wait_metrics: null argument");
  OCF_REQUIRE(step >= 0 && step < m->steps_logged && step + 64 > m->steps_logged, "ocf_model_wait_metrics: step not among the last 64");
  OCF_CUDA(cudaEventSynchronize(m->step_ev[step % 64]));
  std::memcpy(host, m->h_rec + (size_t)(step % LOG_CAP) * LOG_W, sizeof(float) * LOG_W);
  return OCF_OK;
}

static int finish_step(ocf_model* m, float* host_metrics, cudaStream_t) {
  if (host_metrics == nullptr) return OCF_OK;
  return ocf_model_wait_metrics(m, m->steps_logged - 1, host_metrics);
}

// ---- multi-GPU ------------------------------------------------------------------------------------
extern "C" int ocf_comm_unique_id(uint8_t* id) {
  OCF_REQUIRE(id != nullptr, "ocf_comm_unique_id: null argument");
  if (!nccl_api().ok) return fail(OCF_ERR_STATE, "NCCL (libnccl.so.2) could not be loaded");
  ncclUniqueId u;
  OCF_NCCL(nccl_api().getUniqueId(&u));
  std::memcpy(id, u.internal, NCCL_UNIQUE_ID_BYTES);
  return OCF_OK;
}

extern "C" int ocf_comm_destroy(ocf_comm* c);

extern "C" int ocf_comm_info(const ocf_comm* c, int32_t info[3]) {
  OCF_REQUIRE(c && info, "ocf_comm_info: null argument");
  info[0] = c->rank; info[1] = c->world; info[2] = 0;      // [2]: reserved (was: exchanges over peer memory)
  return OCF_OK;
}

extern "C" int ocf_comm_create(const uint8_t* id, int32_t rank, int32_t world, ocf_comm** out) {
  OCF_REQUIRE(id && out && world >= 1 && rank >= 0 && rank < world, "ocf_comm_create: bad argument");
  *out = nullptr;
  if (!nccl_api().ok) return fail(OCF_ERR_STATE, "NCCL (libnccl.so.2) could not be loaded");
  ocf_comm* c = new ocf_comm();
  c->rank = rank; c->world = world;
  if (cudaGetDevice(&c->device) != cudaSuccess) { cudaGetLastError(); delete c; return fail(OCF_ERR_CUDA, "ocf_comm_create: no CUDA device"); }
  ncclUniqueId u;
  std::memcpy(u.internal, id, NCCL_UNIQUE_ID_BYTES);
  ncclResult_t r = nccl_api().commInitRank(&c->comm, world, u, rank);
  if (r != ncclSuccess) { delete c; return fail(OCF_ERR_CUDA, std::string("ncclCommInitRank: ") + nccl_api().getErrorString(r)); }
  g_comms_alive.fetch_add(1);
  *out = c;
  return OCF_OK;
}

extern "C" int ocf_comm_destroy(ocf_comm* c) {
  if (c) {
    cudaDeviceSynchronize();
    if (c->comm) { nccl_api().commDestroy(c->comm); g_comms_alive.fetch_sub(1); }
    delete c;
  }
  return OCF_OK;
}

extern "C" int ocf_model_set_comm(ocf_model* m, ocf_comm* comm, int mode) {
  OCF_REQUIRE(m && (mode == OCF_PAR_COLUMNS || mode == OCF_PAR_ROWS), "ocf_model_set_comm: bad argument");
  OCF_REQUIRE(mode != OCF_PAR_COLUMNS || (comm != nullptr && m->cfg.sharded), "ocf_model_set_comm: column mode needs a communicator and a model created with sharded = 1");
  OCF_REQUIRE(mode != OCF_PAR_ROWS || !m->cfg.sharded, "ocf_model_set_comm: row mode needs an unsharded (replicated) model");
  OCF_CUDA(cudaDeviceSynchronize());
  drop_graphs(m);
  m->comm = comm; m->par_mode = mode;
  if (mode == OCF_PAR_ROWS && m->grads == nullptr) {
    size_t total = 0;
    for (const Layer& ly : m->layers) total += (size_t)ly.rows * ly.hp + (size_t)align_up((size_t)ly.bias_len, 4);
    OCF_TRY(m->par_mem.get(&m->grads, total, true));
    m->grads_count = total;
    m->gW.clear(); m->gb.clear();
    size_t off = 0;
    for (const Layer& ly : m->layers) {
      m->gW.push_back(m->grads + off); off += (size_t)ly.rows * ly.hp;
      m->gb.push_back(m->grads + off); off += align_up((size_t)ly.bias_len, 4);
    }
    const int world = comm ? comm->world : 1;
    OCF_TRY(m->par_mem.get(&m->gathered_stats, (size_t)world * MAX_BATCH_ROWS * ROWSTAT_W, true));
  }
  return OCF_OK;
}

// ---- the two exchanges of a column-sharded step ----------------------------------------------
// phase 1 + exchange of the encoder's partial sums z [rows, H]. *act0_done tells the caller whether launch_act(0) is
// still due (it is: the activation needs the summed z).
static int encode_exchange(ocf_model* m, const ocf_batch* b, bool training, const ocf_step_args* args, cudaStream_t st,
                           bool* act0_done) {
  const int B = b->dev.B;
  *act0_done = false;
  OCF_TRY(phase_encode(m, b, st, nullptr, false, training, args));
  g_prof.begin(6, st);
  OCF_NCCL(nccl_api().allReduce(m->zsum[0], m->zsum[0], (size_t)B * m->hp[0], ncclFloat, ncclSum, m->comm->comm, st));
  g_prof.end(6, st);
  return OCF_OK;
}

// phase 2 + exchange of the row statistics (and dL/dh of the top hidden layer when training).
static int decode_exchange(ocf_model* m, const ocf_batch* b, bool training, const ocf_step_args* args, cudaStream_t st,
                           bool act0_done) {
  const int B = b->dev.B, hpt = m->hp[m->L - 1];
  OCF_TRY(phase_decode(m, b, training, args, nullptr, st, act0_done));
  g_prof.begin(7, st);
  OCF_NCCL(nccl_api().allReduce(m->rowstats, m->rowstats, (size_t)m->cfg.max_rows * ROWSTAT_W + (training ? (size_t)B * hpt : 0),
                                ncclFloat, ncclSum, m->comm->comm, st));
  g_prof.end(7, st);
  return OCF_OK;
}

// Row-parallel mode, after the gradient all-reduce: one streaming pass per parameter array.
static int apply_gradients(ocf_model* m, cudaStream_t st) {
  const OptDev opt = make_opt(m);
  OptDev ob = opt; ob.l2x2 = 0.f;                 // Keras regularises kernels only
  g_prof.begin(6, st);
  for (int l = 0; l <= m->L; ++l) {
    Layer& ly = m->layers[l];
    if (!ly.trainable) continue;
    const size_t n = (size_t)ly.rows * ly.hp;
    const int grid = (int)std::min<size_t>((n / 4 + 255) / 256, (size_t)m->sm_count * 8);
    k_dense_update<<<std::max(grid, 1), 256, 0, st>>>(ly.W, m->gW[l], ly.Ws1, ly.Ws2, n, opt);
    OCF_LAUNCHED();
    k_dense_update<<<std::max(1, std::min((ly.bias_len + 255) / 256, m->sm_count)), 256, 0, st>>>(ly.b, m->gb[l], ly.bs1, ly.bs2, (size_t)ly.bias_len, ob);
    OCF_LAUNCHED();
  }
  g_prof.end(6, st);
  m->iterations += 1;
  return OCF_OK;
}

// Row statistics of the global batch (every rank's rows) for the metrics of a row-parallel step.
static int gather_stats(ocf_model* m, int B, const ocf_step_args* args, const float** stats, int* rows, cudaStream_t st) {
  *stats = m->rowstats; *rows = B;
  if (m->comm == nullptr || m->comm->world == 1) return OCF_OK;
  const int world = m->comm->world;
  OCF_REQUIRE(args && args->rows_total == world * B, "row-parallel step: rows_total must be world x the rank's rows (equal slices)");
  OCF_NCCL(nccl_api().allGather(m->rowstats, m->gathered_stats, (size_t)B * ROWSTAT_W, ncclFloat, m->comm->comm, st));
  *stats = m->gathered_stats; *rows = world * B;
  return OCF_OK;
}

// ---- one step = one body of kernel launches; replayed as a CUDA graph once it has been seen twice ----
// Bodies only enqueue work on `st` (and the side stream forked from it): no allocation, no
// synchronisation, no host-visible bookkeeping, so that they can run under stream capture.
static int train_body(ocf_model* m, ocf_batch* b, const ocf_step_args* args, cudaStream_t st) {
  if (m->par_mode == OCF_PAR_COLUMNS) {
    // column shards: the three phases back to back with the two activation exchanges between them
    // (ncclAllReduce, captured in the step's graph)
    bool act0 = false;
    OCF_TRY(fork_scan(m, b, st));
    OCF_TRY(encode_exchange(m, b, true, args, st, &act0));
    OCF_TRY(decode_exchange(m, b, true, args, st, act0));
    return phase_update(m, b, args, st);
  }
  OCF_TRY(fork_scan(m, b, st));
  OCF_TRY(phase_encode(m, b, st, nullptr, true, true, args));
  OCF_TRY(phase_decode(m, b, true, args, nullptr, st, true, true));
  return phase_update(m, b, args, st, false, nullptr, true);
}

static int eval_body(ocf_model* m, ocf_batch* b, const ocf_step_args* args, cudaStream_t st) {
  if (m->par_mode == OCF_PAR_COLUMNS) {
    bool act0 = false;
    OCF_TRY(encode_exchange(m, b, false, args, st, &act0));
    OCF_TRY(decode_exchange(m, b, false, args, st, act0));
  } else {
    OCF_TRY(phase_encode(m, b, st, nullptr, true, false, args));
    OCF_TRY(phase_decode(m, b, false, args, nullptr, st, true, true));
  }
  const int n_reg = launch_reg(m, st);
  return launch_metrics(m, b->dev.B, args, n_reg, false, st);
}

// ---- K4a ahead of the step --------------------------------------------------------------------------
// The column grouping needs nothing but the gathered batch, so a single-GPU training step runs it on the batch's
// own stream right behind the gather: it executes under whatever step the device is still busy with (the host
// enqueues a step or two ahead) instead of beside this step's K2 / K3.
static bool ahead_ok(const ocf_model* m, const ocf_batch* b, const ocf_step_args* args) {
  return m->par_mode == 0 && m->comm == nullptr && (args == nullptr || args->phase == 0) && b->mode == 1 &&
         b->store != nullptr && b->gathered_valid &&
         (m->layers[0].trainable || m->layers[m->L].trainable) && b->dev.B <= b->max_rows;
}

// [seg | counters | state | bits] is one region: a single memset clears what K4a counts into.
static int worklist_alloc(ocf_batch* b, const ocf_model* m) {
  const size_t N = (size_t)m->cfg.n_cols;
  if (b->wl_cols == m->cfg.n_cols && b->wl_nblk == m->nblk) return OCF_OK;
  if (b->wl_cols != 0) {
    // another catalogue / input layout: steps captured with the old pointers are stale, the batch takes a new identity
    OCF_CUDA(cudaDeviceSynchronize());
    b->wl_mem.release();
    if (b->wl_graph) { cudaGraphExecDestroy(b->wl_graph); b->wl_graph = nullptr; }
    b->wl_graph_failed = false;
    b->uid = ++g_batch_uid;
    b->wl_cols = 0; b->wl_seq = 0;
  }
  const size_t Wcap = (size_t)(b->max_rows + 31) / 32;
  const size_t seg_b = sizeof(int2) * N, cnt_b = 32, state_b = sizeof(int) * 2 * N, bits_b = sizeof(uint32_t) * N * Wcap;
  uint8_t* z = nullptr;
  OCF_TRY(b->wl_mem.get(&z, seg_b + cnt_b + state_b + bits_b, true));
  b->wl_zero = z;
  b->wl.seg = reinterpret_cast<int2*>(z);
  b->wl.counters = reinterpret_cast<int*>(z + seg_b);
  b->wl.state = reinterpret_cast<int*>(z + seg_b + cnt_b);
  b->wl.bits = reinterpret_cast<uint32_t*>(z + seg_b + cnt_b + state_b);
  OCF_TRY(b->wl_mem.get(&b->wl.tasks, N * (size_t)(m->nblk + 1)));
  OCF_TRY(b->wl_mem.get(&b->wl.heavy, N * (size_t)(m->nblk + 1)));
  OCF_TRY(b->wl_mem.get(&b->wl.info, N));
  OCF_TRY(b->wl_mem.get(&b->wl.matches, (size_t)std::max<int64_t>(b->max_entries, 1) * 3));
  b->wl.entries = b->max_entries;
  b->wl_cols = m->cfg.n_cols; b->wl_nblk = m->nblk;
  return OCF_OK;
}

static int worklist_enqueue(ocf_model* m, ocf_batch* b, const WorkSig& sig, cudaStream_t s) {
  const size_t N = (size_t)sig.n_cols, W = (size_t)(sig.B + 31) / 32;
  uint8_t* z0 = sig.dense ? b->wl_zero : reinterpret_cast<uint8_t*>(b->wl.counters);
  const size_t bytes = (sig.dense ? sizeof(int2) * N : 0) + 32 + sizeof(int) * 2 * N + sizeof(uint32_t) * N * W;
  OCF_CUDA(cudaMemsetAsync(z0, 0, bytes, s));
  return launch_scan(m, b, sig.do_dec, sig.do_enc, sig.dense, s, b->wl, true);
}

static int prepare_worklist(ocf_model* m, ocf_batch* b, cudaStream_t user) {
  const WorkSig sig = work_sig(m, b);
  if (b->wl_seq != 0 && b->wl_seq == b->fill_seq && b->wl_sig == sig) {
    // a second step on the same fill walks the same list: only K4b's task cursors start over
    OCF_CUDA(cudaMemsetAsync(b->wl.counters + 3, 0, 2 * sizeof(int), user));
    return OCF_OK;
  }
  OCF_TRY(worklist_alloc(b, m));
  cudaStream_t gs = b->gstream;                                                        // the fill ran here: in order behind it
  if (b->consumed_valid) OCF_CUDA(cudaStreamWaitEvent(gs, b->consumed, 0));            // the list's previous reader
  bool done = false;
  if (!g_prof.on) {
    if (b->wl_graph != nullptr && !(b->wl_graph_sig == sig)) { cudaGraphExecDestroy(b->wl_graph); b->wl_graph = nullptr; b->wl_graph_failed = false; }
    if (b->wl_graph == nullptr && !b->wl_graph_failed) {
      const long long launched = g_launches.load();
      const bool was_capturing = m->capturing;
      m->capturing = true;                         // grids sized to the batch object's capacity (item_grid)
      cudaGraph_t graph = nullptr;
      int rc = OCF_OK;
      // captured kernel nodes inherit the capture stream's priority: m->cap runs at the batch streams' (the highest)
      if (cudaStreamBeginCapture(m->cap, cudaStreamCaptureModeThreadLocal) != cudaSuccess) { cudaGetLastError(); rc = OCF_ERR_CUDA; }
      else {
        rc = worklist_enqueue(m, b, sig, m->cap);
        if (cudaStreamEndCapture(m->cap, &graph) != cudaSuccess) { cudaGetLastError(); rc = OCF_ERR_CUDA; graph = nullptr; }
      }
      m->capturing = was_capturing;
      b->wl_graph_kernels = (int)(g_launches.load() - launched);
      g_launches.store(launched);
      if (rc == OCF_OK && graph != nullptr && cudaGraphInstantiate(&b->wl_graph, graph, 0) != cudaSuccess) { cudaGetLastError(); b->wl_graph = nullptr; }
      if (graph) cudaGraphDestroy(graph);
      if (b->wl_graph == nullptr) b->wl_graph_failed = true; else b->wl_graph_sig = sig;
    }
    if (b->wl_graph != nullptr) {
      OCF_CUDA(cudaGraphLaunch(b->wl_graph, gs));
      g_launches.fetch_add(b->wl_graph_kernels, std::memory_order_relaxed);
      done = true;
    }
  }
  if (!done) OCF_TRY(worklist_enqueue(m, b, sig, gs));
  OCF_CUDA(cudaEventRecord(b->wl_ready, gs));
  b->wl_seq = b->fill_seq; b->wl_sig = sig;
  return OCF_OK;
}

// Runs a whole step (phase 0) of a single-GPU or column-sharded model. The first time a (batch object,
// rows, kind) combination is seen the body runs as plain launches (lazy allocations happen there), the
// second time it is captured into a CUDA graph, from then on the graph is replayed: one launch per step,
// every size and scalar that changes from step to step is read from device memory (BatchHdr, StepDev).
static int run_step(ocf_model* m, ocf_batch* b, const ocf_step_args* args, bool train, cudaStream_t st) {
  OCF_TRY(sync_step_state(m, args, st));
  auto body = [&](cudaStream_t s) { return train ? train_body(m, b, args, s) : eval_body(m, b, args, s); };
  bool done = false;
  if (!g_prof.on) {
    const auto key = std::make_tuple(b->uid, b->dev.B, train ? (wl_current(m, b) ? 3 : 1) : 0, args ? args->rows_total : 0, args ? args->row0 : 0,
                                     b->store->has_dups ? 1 : 0);
    ocf_model::StepGraph& g = m->graphs[key];
    if (g.exec == nullptr && !g.failed && g.seen++ >= 1) {
      const long long launched = g_launches.load();
      m->capturing = true;
      cudaGraph_t graph = nullptr;
      int rc = OCF_OK;
      if (cudaStreamBeginCapture(m->cap, cudaStreamCaptureModeThreadLocal) != cudaSuccess) { cudaGetLastError(); rc = OCF_ERR_CUDA; }
      else {
        rc = body(m->cap);
        if (cudaStreamEndCapture(m->cap, &graph) != cudaSuccess) { cudaGetLastError(); rc = OCF_ERR_CUDA; graph = nullptr; }
      }
      m->capturing = false;
      m->scan_pending = false;
      g.kernels = (int)(g_launches.load() - launched);
      g_launches.store(launched);
      if (rc == OCF_OK && graph != nullptr && cudaGraphInstantiate(&g.exec, graph, 0) != cudaSuccess) { cudaGetLastError(); g.exec = nullptr; }
      if (graph) cudaGraphDestroy(graph);
      if (g.exec == nullptr) {                         // this combination keeps running as plain launches
        g.failed = true;
        if (std::getenv("OCF_DEBUG_GRAPH")) std::fprintf(stderr, "[ocf] step graph capture failed (rc %d): plain launches from here on\n", rc);
      } else if (std::getenv("OCF_DEBUG_GRAPH")) {
        std::fprintf(stderr, "[ocf] step graph captured: %d kernels\n", g.kernels);
      }
    }
    if (g.exec != nullptr) {
      OCF_CUDA(cudaGraphLaunch(g.exec, st));
      g_launches.fetch_add(g.kernels, std::memory_order_relaxed);
      done = true;
    }
  }
  if (!done) OCF_TRY(body(st));
  if (train) m->iterations += 1;
  return publish_metrics(m, train, st);
}

static int ocf_train_step_impl(ocf_model* m, ocf_batch* b, const ocf_step_args* args, float* host_metrics, void* stream_);
extern "C" int ocf_train_step(ocf_model* m, ocf_batch* b, const ocf_step_args* args, float* host_metrics, void* stream_) {
  if (m && b && check_step(m, b, true) == OCF_OK && ahead_ok(m, b, args)) OCF_TRY(prepare_worklist(m, b, as_stream(stream_)));
  if (b) OCF_TRY(batch_acquire(b, as_stream(stream_)));          // the batch's fill runs on its own stream
  if (m && b && wl_current(m, b)) OCF_CUDA(cudaStreamWaitEvent(as_stream(stream_), b->wl_ready, 0));
  const int rc = ocf_train_step_impl(m, b, args, host_metrics, stream_);
  if (b && rc == OCF_OK) OCF_TRY(batch_release(b, as_stream(stream_)));
  return rc;
}
static int ocf_train_step_impl(ocf_model* m, ocf_batch* b, const ocf_step_args* args, float* host_metrics, void* stream_) {
  OCF_TRY(check_step(m, b, true));
  cudaStream_t st = as_stream(stream_);
  const int phase = args ? args->phase : 0;
  OCF_REQUIRE(phase >= 0 && phase <= 3, "ocf_train_step: phase must be 0..3");
  if (phase == 0 && m->par_mode == OCF_PAR_ROWS) {
    // data parallel over rows: replicated weights, this rank's rows, gradients summed over ranks
    OCF_TRY(sync_step_state(m, args, st));
    OCF_TRY(fork_scan(m, b, st));
    OCF_TRY(phase_encode(m, b, st, nullptr, true, true, args));
    OCF_TRY(phase_decode(m, b, true, args, nullptr, st, true));
    int n_reg = 0;
    OCF_TRY(phase_update(m, b, args, st, true, &n_reg));
    if (m->comm && m->comm->world > 1) {
      g_prof.begin(7, st);
      OCF_NCCL(nccl_api().allReduce(m->grads, m->grads, m->grads_count, ncclFloat, ncclSum, m->comm->comm, st));
      g_prof.end(7, st);
    }
    const float* stats; int rows;
    OCF_TRY(gather_stats(m, b->dev.B, args, &stats, &rows, st));
    OCF_TRY(apply_gradients(m, st));
    OCF_TRY(launch_metrics(m, rows, args, n_reg, true, st, stats));
    OCF_TRY(publish_metrics(m, true, st));
    return finish_step(m, host_metrics, st);
  }
  if (phase == 0) {
    OCF_TRY(run_step(m, b, args, true, st));
    return finish_step(m, host_metrics, st);
  }
  // a step driven phase by phase (a caller that runs the shard exchanges itself between the phases)
  OCF_TRY(sync_step_state(m, args, st));
  if (phase == 1) { OCF_TRY(fork_scan(m, b, st)); OCF_TRY(phase_encode(m, b, st, nullptr, false, true, args)); }
  if (phase == 2) OCF_TRY(phase_decode(m, b, true, args, nullptr, st));
  if (phase == 3) {
    OCF_TRY(phase_update(m, b, args, st));
    m->iterations += 1;
    OCF_TRY(publish_metrics(m, true, st));
    OCF_TRY(finish_step(m, host_metrics, st));
  }
  return OCF_OK;
}

static int ocf_eval_step_impl(ocf_model* m, ocf_batch* b, const ocf_step_args* args, float* host_metrics, void* stream_);
extern "C" int ocf_eval_step(ocf_model* m, ocf_batch* b, const ocf_step_args* args, float* host_metrics, void* stream_) {
  if (b) OCF_TRY(batch_acquire(b, as_stream(stream_)));          // the batch's fill runs on its own stream
  const int rc = ocf_eval_step_impl(m, b, args, host_metrics, stream_);
  if (b && rc == OCF_OK) OCF_TRY(batch_release(b, as_stream(stream_)));
  return rc;
}
static int ocf_eval_step_impl(ocf_model* m, ocf_batch* b, const ocf_step_args* args, float* host_metrics, void* stream_) {
  OCF_TRY(check_step(m, b, false));
  cudaStream_t st = as_stream(stream_);
  const int phase = args ? args->phase : 0;
  OCF_REQUIRE(phase >= 0 && phase <= 3, "ocf_eval_step: phase must be 0..3");
  if (phase == 0 && m->par_mode == OCF_PAR_ROWS) {
    OCF_TRY(sync_step_state(m, args, st));
    OCF_TRY(phase_encode(m, b, st, nullptr, true, false, args));
    OCF_TRY(phase_decode(m, b, false, args, nullptr, st, true));
    const float* stats; int rows;
    OCF_TRY(gather_stats(m, b->dev.B, args, &stats, &rows, st));
    const int n_reg = launch_reg(m, st);
    OCF_TRY(launch_metrics(m, rows, args, n_reg, false, st, stats));
    OCF_TRY(publish_metrics(m, false, st));
    return finish_step(m, host_metrics, st);
  }
  if (phase == 0) {
    OCF_TRY(run_step(m, b, args, false, st));
    return finish_step(m, host_metrics, st);
  }
  OCF_TRY(sync_step_state(m, args, st));
  if (phase == 1) OCF_TRY(phase_encode(m, b, st, nullptr, false, false, args));
  if (phase == 2) OCF_TRY(phase_decode(m, b, false, args, nullptr, st));
  if (phase == 3) {
    const int n_reg = launch_reg(m, st);
    OCF_TRY(launch_metrics(m, b->dev.B, args, n_reg, false, st));
    OCF_TRY(publish_metrics(m, false, st));
    OCF_TRY(finish_step(m, host_metrics, st));
  }
  return OCF_OK;
}

// Encoder pre-activations for predict / score. A column shard with a communicator reduces them
// here; without one its caller has already run phase 1 and the z all-reduce.
static int encode_for_output(ocf_model* m, const ocf_batch* b, cudaStream_t st, bool* act0_done) {
  *act0_done = false;
  OCF_TRY(sync_step_state(m, nullptr, st));
  if (!m->cfg.sharded) { *act0_done = true; return phase_encode(m, b, st, nullptr, true, false, nullptr); }
  if (m->par_mode == OCF_PAR_COLUMNS) return encode_exchange(m, b, false, nullptr, st, act0_done);
  return OCF_OK;
}

static int ensure_dense(ocf_model* m) {
  if (m->dense_out) return OCF_OK;
  return m->dense_mem.get(&m->dense_out, (size_t)m->cfg.max_rows * m->cfg.n_cols);
}

static int ocf_predict_impl(ocf_model* m, ocf_batch* b, float* out, void* stream_);
extern "C" int ocf_predict(ocf_model* m, ocf_batch* b, float* out, void* stream_) {
  if (b) OCF_TRY(batch_acquire(b, as_stream(stream_)));          // the batch's fill runs on its own stream
  const int rc = ocf_predict_impl(m, b, out, stream_);
  if (b && rc == OCF_OK) OCF_TRY(batch_release(b, as_stream(stream_)));
  return rc;
}
static int ocf_predict_impl(ocf_model* m, ocf_batch* b, float* out, void* stream_) {
  OCF_TRY(check_step(m, b, false));
  OCF_REQUIRE(out != nullptr, "ocf_predict: null output");
  cudaStream_t st = as_stream(stream_);
  OCF_TRY(ensure_dense(m));
  const size_t count = (size_t)b->dev.B * m->cfg.n_cols;
  OCF_CUDA(cudaMemsetAsync(m->dense_out, 0, sizeof(float) * count, st));
  bool act0 = false;
  OCF_TRY(encode_for_output(m, b, st, &act0));
  OCF_TRY(phase_decode(m, b, false, nullptr, m->dense_out, st, act0));
  OCF_CUDA(cudaMemcpyAsync(out, m->dense_out, sizeof(float) * count, cudaMemcpyDeviceToHost, st));
  OCF_CUDA(cudaStreamSynchronize(st));
  return OCF_OK;
}

static int ocf_score_impl(ocf_model* m, ocf_batch* b, float* out, int out_is_device, void* stream_);
extern "C" int ocf_score(ocf_model* m, ocf_batch* b, float* out, int out_is_device, void* stream_) {
  if (b) OCF_TRY(batch_acquire(b, as_stream(stream_)));          // the batch's fill runs on its own stream
  const int rc = ocf_score_impl(m, b, out, out_is_device, stream_);
  if (b && rc == OCF_OK) OCF_TRY(batch_release(b, as_stream(stream_)));
  return rc;
}
static int ocf_score_impl(ocf_model* m, ocf_batch* b, float* out, int out_is_device, void* stream_) {
  OCF_TRY(check_step(m, b, false));
  OCF_REQUIRE(out != nullptr, "ocf_score: null output");
  cudaStream_t st = as_stream(stream_);
  const int L = m->L, B = b->dev.B;
  bool act0 = false;
  OCF_TRY(encode_for_output(m, b, st, &act0));
  if (!act0) OCF_TRY(launch_act(m, 0, B, false, nullptr, st));
  for (int l = 1; l < L; ++l) OCF_TRY(hidden_fwd_tc(m, l, B, m->act[l - 1], act_args(m, l, B, false, nullptr), st));
  float* dst = out;
  if (!out_is_device) { OCF_TRY(ensure_dense(m)); dst = m->dense_out; }
  // decoder GEMM on the tensor cores: tcgen05.mma kind::tf32, accumulators in TMEM (ocf_score_tc.cuh)
  const Layer& dec = m->layers[L];
  const int hpt = m->hp[L - 1];
  if (!m->map_w_ok) {
    OCF_TRY(tc::make_map(&m->map_w, dec.W, hpt, (long long)align_up((size_t)m->cfg.n_cols, 2 * tc::TILE_M), tc::TILE_M));
    m->map_w_ok = true;
  }
  const int nb = tc::chunk_rows(B);
  const int box = nb / 2;                         // a CTA of a pair loads half of the batch-row operand
  if (!m->map_h_ok || m->map_h_box != box) {
    OCF_TRY(tc::make_map(&m->map_h, m->act[L - 1], hpt, m->act_rows, box));
    m->map_h_ok = true; m->map_h_box = box;
  }
  tc::ScoreArgs sa{};
  sa.bias = dec.b; sa.out = dst; sa.ldo = m->cfg.n_cols; sa.n_cols = m->cfg.n_cols; sa.n_rows = B;
  sa.num_k = hpt / tc::BLOCK_K; sa.n_mtiles = (m->cfg.n_cols + tc::TILE_M - 1) / tc::TILE_M; sa.n_chunks = (B + nb - 1) / nb;
  g_prof.begin(4, st);
  if (nb == 64) OCF_TRY(tc::launch_score_pair_nb<64>(m->map_w, m->map_h, sa, m->sm_count, st));
  else if (nb == 128) OCF_TRY(tc::launch_score_pair_nb<128>(m->map_w, m->map_h, sa, m->sm_count, st));
  else OCF_TRY(tc::launch_score_pair_nb<256>(m->map_w, m->map_h, sa, m->sm_count, st));
  g_prof.end(4, st);
  if (!out_is_device) {
    OCF_CUDA(cudaMemcpyAsync(out, dst, sizeof(float) * (size_t)B * m->cfg.n_cols, cudaMemcpyDeviceToHost, st));
    OCF_CUDA(cudaStreamSynchronize(st));
  }
  return OCF_OK;
}

// The full-catalogue scores of the batch into dense_out (they stay in HBM), the row's input columns set
// to -inf when `exclude_inputs`: what the serving epilogues (top-k, ranking evaluation) read.
static int score_to_dense(ocf_model* m, ocf_batch* b, int exclude_inputs, void* stream_) {
  cudaStream_t st = as_stream(stream_);
  OCF_TRY(ensure_dense(m));
  OCF_TRY(ocf_score(m, b, m->dense_out, 1, stream_));
  if (exclude_inputs && b->dev.n_items > 0) {
    k_exclude_inputs<<<b->dev.n_items, 128, 0, st>>>(b->dev, m->dense_out, (long long)m->cfg.n_cols);
    OCF_LAUNCHED();
  }
  return OCF_OK;
}

static int ocf_score_topk_impl(ocf_model* m, ocf_batch* b, int32_t k, int exclude_inputs, int32_t* out_cols, float* out_scores,
                              void* stream_);
extern "C" int ocf_score_topk(ocf_model* m, ocf_batch* b, int32_t k, int exclude_inputs, int32_t* out_cols, float* out_scores,
                              void* stream_) {
  if (b) OCF_TRY(batch_acquire(b, as_stream(stream_)));
  const int rc = ocf_score_topk_impl(m, b, k, exclude_inputs, out_cols, out_scores, stream_);
  if (b && rc == OCF_OK) OCF_TRY(batch_release(b, as_stream(stream_)));
  return rc;
}
static int ocf_score_topk_impl(ocf_model* m, ocf_batch* b, int32_t k, int exclude_inputs, int32_t* out_cols, float* out_scores,
                              void* stream_) {
  OCF_TRY(check_step(m, b, false));
  OCF_REQUIRE(out_cols && out_scores, "ocf_score_topk: null output");
  OCF_REQUIRE(k >= 1 && k <= TOPK_MAX, "ocf_score_topk: k must be in 1..512");
  cudaStream_t st = as_stream(stream_);
  const int B = b->dev.B;
  OCF_TRY(ensure_dense(m));
  if (m->topk_cap < (size_t)m->cfg.max_rows * TOPK_MAX) {
    OCF_TRY(m->dense_mem.get(&m->topk_cols, (size_t)m->cfg.max_rows * TOPK_MAX));
    OCF_TRY(m->dense_mem.get(&m->topk_scores, (size_t)m->cfg.max_rows * TOPK_MAX));
    m->topk_cap = (size_t)m->cfg.max_rows * TOPK_MAX;
  }
  OCF_TRY(score_to_dense(m, b, exclude_inputs, stream_));
  g_prof.begin(6, st);
  k_topk<<<B, TOPK_THREADS, 0, st>>>(m->dense_out, (long long)m->cfg.n_cols, m->cfg.n_cols, k, m->topk_cols, m->topk_scores);
  OCF_LAUNCHED();
  g_prof.end(6, st);
  OCF_CUDA(cudaMemcpyAsync(out_cols, m->topk_cols, sizeof(int32_t) * (size_t)B * k, cudaMemcpyDeviceToHost, st));
  OCF_CUDA(cudaMemcpyAsync(out_scores, m->topk_scores, sizeof(float) * (size_t)B * k, cudaMemcpyDeviceToHost, st));
  OCF_CUDA(cudaStreamSynchronize(st));
  return OCF_OK;
}

static int ocf_rank_targets_impl(ocf_model* m, ocf_batch* b, int exclude_inputs, float min_value, int32_t* out_col,
                                 int32_t* out_rank, int32_t* out_row_ptr, int64_t* out_n_cand, void* stream_);
extern "C" int ocf_rank_targets(ocf_model* m, ocf_batch* b, int exclude_inputs, float min_value, int32_t* out_col,
                                int32_t* out_rank, int32_t* out_row_ptr, int64_t* out_n_cand, void* stream_) {
  if (b) OCF_TRY(batch_acquire(b, as_stream(stream_)));
  const int rc = ocf_rank_targets_impl(m, b, exclude_inputs, min_value, out_col, out_rank, out_row_ptr, out_n_cand, stream_);
  if (b && rc == OCF_OK) OCF_TRY(batch_release(b, as_stream(stream_)));
  return rc;
}
static int ocf_rank_targets_impl(ocf_model* m, ocf_batch* b, int exclude_inputs, float min_value, int32_t* out_col,
                                 int32_t* out_rank, int32_t* out_row_ptr, int64_t* out_n_cand, void* stream_) {
  OCF_TRY(check_step(m, b, false));
  OCF_REQUIRE(out_col && out_rank && out_row_ptr && out_n_cand, "ocf_rank_targets: null output");
  OCF_REQUIRE(!m->cfg.sharded && m->par_mode != OCF_PAR_COLUMNS,
              "ocf_rank_targets: a column shard holds part of the catalogue; ranks need every column");
  cudaStream_t st = as_stream(stream_);
  const int B = b->dev.B, E = b->dev.n_entries;
  OCF_TRY(ensure_dense(m));
  if (!m->rank_ok) {
    const size_t cap = (size_t)std::max<int64_t>(m->cfg.max_entries, 1);
    OCF_TRY(m->dense_mem.get(&m->rank_key, cap));
    OCF_TRY(m->dense_mem.get(&m->rank_col, cap));
    OCF_TRY(m->dense_mem.get(&m->rank_ent, cap));
    OCF_TRY(m->dense_mem.get(&m->rank_cnt, cap));
    OCF_TRY(m->dense_mem.get(&m->rank_out, cap));
    OCF_TRY(m->dense_mem.get(&m->rank_nrel, (size_t)m->cfg.max_rows));
    OCF_TRY(m->dense_mem.get(&m->rank_ncand, (size_t)m->cfg.max_rows));
    m->rank_ok = true;
  }
  OCF_TRY(score_to_dense(m, b, exclude_inputs, stream_));
  RankArgs ra{};
  ra.bt = b->dev; ra.scores = m->dense_out; ra.ldo = m->cfg.n_cols; ra.n_cols = m->cfg.n_cols; ra.min_value = min_value;
  ra.key = m->rank_key; ra.col = m->rank_col; ra.ent = m->rank_ent; ra.cnt = m->rank_cnt;
  ra.n_rel = m->rank_nrel; ra.n_cand = m->rank_ncand; ra.rank = m->rank_out;
  // enough column slices that even a batch of one row spreads over every SM, none shorter than 4096 columns
  const int N = m->cfg.n_cols;
  const int want = (16 * m->sm_count + B - 1) / B;
  const int slices = std::max(1, std::min(want, (N + 4095) / 4096));
  ra.slice_len = (int)align_up((size_t)((N + slices - 1) / slices), 4);
  const int grid_x = (N + ra.slice_len - 1) / ra.slice_len;
  if (B > 0) {
    g_prof.begin(9, st);
    k_rank_prep<<<B, RANK_THREADS, 0, st>>>(ra);
    OCF_LAUNCHED();
    k_rank_count<<<dim3(grid_x, B), RANK_THREADS, 0, st>>>(ra);
    OCF_LAUNCHED();
    k_rank_finish<<<B, RANK_THREADS, 0, st>>>(ra);
    OCF_LAUNCHED();
    g_prof.end(9, st);
  }
  static_assert(sizeof(unsigned long long) == sizeof(int64_t), "n_cand is copied as int64");
  if (E > 0) {
    OCF_CUDA(cudaMemcpyAsync(out_col, b->dev.ent_col, sizeof(int32_t) * (size_t)E, cudaMemcpyDeviceToHost, st));
    OCF_CUDA(cudaMemcpyAsync(out_rank, m->rank_out, sizeof(int32_t) * (size_t)E, cudaMemcpyDeviceToHost, st));
  }
  OCF_CUDA(cudaMemcpyAsync(out_row_ptr, b->dev.ent_off, sizeof(int32_t) * (size_t)(B + 1), cudaMemcpyDeviceToHost, st));
  if (B > 0) OCF_CUDA(cudaMemcpyAsync(out_n_cand, m->rank_ncand, sizeof(int64_t) * (size_t)B, cudaMemcpyDeviceToHost, st));
  OCF_CUDA(cudaStreamSynchronize(st));
  return OCF_OK;
}

extern "C" int ocf_gemm_tc(const float* a, int a_mn, const float* b, int b_mn, int32_t m_len, int32_t n_len, int32_t k_len,
                           int terms, int split, float* out) {
  OCF_REQUIRE(a && b && out && m_len > 0 && n_len > 0 && k_len > 0, "ocf_gemm_tc: bad argument");
  OCF_REQUIRE(m_len % 4 == 0 && n_len % 4 == 0 && k_len % 4 == 0, "ocf_gemm_tc: sizes must be multiples of 4 (16-byte rows for TMA)");
  OCF_REQUIRE(terms == 1 || terms == 3, "ocf_gemm_tc: terms must be 1 or 3");
  OCF_REQUIRE(split == 0 || split == 1 || split == 2 || split == 4 || split == 8, "ocf_gemm_tc: split must be 0, 1, 2, 4 or 8");
  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) { cudaGetLastError(); return fail(OCF_ERR_CUDA, "ocf_gemm_tc: no CUDA device"); }
  Arena mem;
  struct Release { Arena& a; ~Release() { a.release(); } } release_on_exit{mem};
  float *da = nullptr, *db = nullptr, *dc = nullptr;
  const size_t na = (size_t)m_len * k_len, nb = (size_t)n_len * k_len, nc = (size_t)m_len * n_len;
  OCF_TRY(mem.get(&da, na)); OCF_TRY(mem.get(&db, nb)); OCF_TRY(mem.get(&dc, nc, true));
  OCF_CUDA(cudaMemcpy(da, a, na * sizeof(float), cudaMemcpyHostToDevice));
  OCF_CUDA(cudaMemcpy(db, b, nb * sizeof(float), cudaMemcpyHostToDevice));
  CUtensorMap ma, mb;
  if (a_mn) OCF_TRY(gtc::make_map_mn(&ma, da, m_len, m_len, k_len)); else OCF_TRY(gtc::make_map_k(&ma, da, k_len, k_len, m_len));
  if (b_mn) OCF_TRY(gtc::make_map_mn(&mb, db, n_len, n_len, k_len)); else OCF_TRY(gtc::make_map_k(&mb, db, k_len, k_len, n_len));
  gtc::GemmTcArgs g{};
  g.kind = gtc::GEPI_RAW; g.a_mn = a_mn ? 1 : 0; g.b_mn = b_mn ? 1 : 0; g.C = dc; g.ldc = m_len; g.terms = terms;
  OCF_TRY(gtc::launch(ma, mb, g, m_len, n_len, k_len, nullptr, split));
  OCF_CUDA(cudaDeviceSynchronize());
  OCF_CUDA(cudaMemcpy(out, dc, nc * sizeof(float), cudaMemcpyDeviceToHost));
  return OCF_OK;
}

// Diagnostic twin of ocf_gemm_tc: `reps` launches of the update-kind contraction (read-modify-write epilogue) on
// device-resident random operands, CUDA-event time per launch and the phase stamps of CTA (0,0,0) of the last launch.
extern "C" int ocf_gemm_tc_profile(int a_mn, int b_mn, int32_t m_len, int32_t n_len, int32_t k_len, int split, int kind, int reps,
                                   float* ms_per_launch, int64_t stamps_ns[8]) {
  OCF_REQUIRE(ms_per_launch && stamps_ns && reps > 0, "ocf_gemm_tc_profile: bad argument");
  Arena mem;
  struct Release { Arena& a; ~Release() { a.release(); } } release_on_exit{mem};
  float *da = nullptr, *db = nullptr, *dc = nullptr, *ds = nullptr, *dx = nullptr;
  unsigned long long* dbg = nullptr;
  const size_t na = (size_t)m_len * k_len, nb = (size_t)n_len * k_len, nc = (size_t)m_len * n_len;
  OCF_TRY(mem.get(&da, na, true)); OCF_TRY(mem.get(&db, nb, true)); OCF_TRY(mem.get(&dc, nc, true)); OCF_TRY(mem.get(&ds, nc, true));
  OCF_TRY(mem.get(&dx, nc, true)); OCF_TRY(mem.get(&dbg, 8, true));
  StepDev* dstep = nullptr;
  OCF_TRY(mem.get(&dstep, 1, true));
  CUtensorMap ma, mb;
  if (a_mn) OCF_TRY(gtc::make_map_mn(&ma, da, m_len, m_len, k_len)); else OCF_TRY(gtc::make_map_k(&ma, da, k_len, k_len, m_len));
  if (b_mn) OCF_TRY(gtc::make_map_mn(&mb, db, n_len, n_len, k_len)); else OCF_TRY(gtc::make_map_k(&mb, db, k_len, k_len, n_len));
  gtc::GemmTcArgs g{};
  g.kind = kind; g.a_mn = a_mn ? 1 : 0; g.b_mn = b_mn ? 1 : 0; g.C = dc; g.ldc = m_len; g.terms = 3; g.dbg = dbg;
  g.s1 = ds; g.aux0 = dx; g.act = OCF_ACT_SIGMOID;
  g.opt.kind = OCF_OPT_ADAGRAD; g.opt.eps = 1e-8f; g.opt.st = dstep;
  cudaEvent_t e0, e1;
  OCF_CUDA(cudaEventCreate(&e0)); OCF_CUDA(cudaEventCreate(&e1));
  for (int i = 0; i < 3; ++i) OCF_TRY(gtc::launch(ma, mb, g, m_len, n_len, k_len, nullptr, split));
  OCF_CUDA(cudaEventRecord(e0, nullptr));
  for (int i = 0; i < reps; ++i) OCF_TRY(gtc::launch(ma, mb, g, m_len, n_len, k_len, nullptr, split));
  OCF_CUDA(cudaEventRecord(e1, nullptr));
  OCF_CUDA(cudaDeviceSynchronize());
  float ms = 0.f;
  OCF_CUDA(cudaEventElapsedTime(&ms, e0, e1));
  *ms_per_launch = ms / reps;
  unsigned long long h[8];
  OCF_CUDA(cudaMemcpy(h, dbg, sizeof(h), cudaMemcpyDeviceToHost));
  for (int i = 0; i < 8; ++i) stamps_ns[i] = (int64_t)(h[i] - h[0]);
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  return OCF_OK;
}

extern "C" int ocf_model_read_metrics(ocf_model* m, int64_t first, int32_t count, float* host, void* stream_) {
  OCF_REQUIRE(m && host, "ocf_model_read_metrics: null argument");
  OCF_REQUIRE(count >= 0 && count <= LOG_CAP && first >= 0 && first + count <= m->steps_logged &&
              first + LOG_CAP >= m->steps_logged, "ocf_model_read_metrics: range not in the log");
  cudaStream_t st = as_stream(stream_);
  OCF_CUDA(cudaStreamSynchronize(st));
  if (m->steps_logged > 0) OCF_CUDA(cudaEventSynchronize(m->step_ev[(m->steps_logged - 1) % 64]));
  for (int32_t k = 0; k < count; ++k)
    std::memcpy(host + (size_t)k * LOG_W, m->h_rec + (size_t)((first + k) % LOG_CAP) * LOG_W, sizeof(float) * LOG_W);
  return OCF_OK;
}
