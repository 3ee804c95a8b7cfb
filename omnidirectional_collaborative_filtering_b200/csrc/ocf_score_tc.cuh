// Full-catalogue scoring on the 5th-generation tensor cores (tcgen05 + TMEM + TMA), sm_100a only.
//
//   full[b, c] = sum_k h[b, k] * WdecT[c, k] + bias[c]          (model.py:82-84, before the mask)
//
// The catalogue runs along the MMA's M (128 TMEM lanes), the batch rows along N, so one TMEM
// column is one batch row and a warp's 32 lanes are 32 consecutive catalogue columns: the
// epilogue's stores are 128-byte coalesced without a shared-memory transpose.  Both operands are
// K-major in HBM already (WdecT [N, hp] and h [rows, hp], fp32 read as tf32), so TMA drops
// 128-byte-swizzled [rows x 32] boxes straight into the layout the MMA descriptors name.
//
// Warp roles (320 threads): warp 0 = TMA producer (one elected lane), warp 1 = TMEM owner + MMA
// issuer (one elected lane), warps 2..9 = epilogue (TMEM -> registers -> +bias -> HBM).  Two accumulator stages
// in TMEM let the epilogue of tile t overlap the MMAs of tile t+1; a ring of smem stages
// decouples TMA from the MMAs.  Persistent: at most one CTA pair per two SMs, tiles strided over the pairs.
#pragma once

#include <cuda.h>

#include "ocf_common.cuh"

namespace ocf {
namespace tc {

constexpr int TILE_M = 128;    // catalogue columns per tile = UMMA M
constexpr int BLOCK_K = 32;    // tf32 elements per 128-byte swizzle row
constexpr int UMMA_K = 8;      // tf32 elements one tcgen05.mma consumes along K (32 bytes)
constexpr int EPI_WARPS = 8;    // two warps per TMEM lane quarter, each draining every other 32-row chunk
constexpr int NTHREADS = 64 + 32 * EPI_WARPS;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must end in a trapped launch, not in a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) asm volatile("trap;");
  }
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// One lane of a converged warp (the warp stays converged around the elected work, so the
// barrier waits and loop counters run on the uniform datapath: a role loop written under
// `if (lane == 0)` made the single issuing thread the bottleneck - ~1650 cycles per k-block of
// scalarised descriptor moves against 512 cycles of tensor work, profiles/r01 score v2).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// Shared-memory matrix descriptor of a K-major, 128-byte-swizzled [rows x 32 tf32] box: 8-row
// groups are 1024 bytes apart (SBO), the leading offset is unused under swizzle (1), version 1
// (Blackwell), layout type 2 (SWIZZLE_128B).
__device__ __forceinline__ uint64_t make_desc(const void* smem_ptr) {
  const uint32_t a = smem_u32(smem_ptr);
  uint64_t d = 0;
  d |= (uint64_t)((a >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrives on the mbarrier once every MMA issued so far by this thread has completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// One TMEM chunk of a warp: register i of every lane belongs to batch row i, the lanes are 32
// consecutive catalogue columns: 32 stores of 128 contiguous bytes each. The full chunk is
// straight-line predicated code (a per-row `if` inside the unrolled loop cost a reconvergence
// barrier per store and capped the whole kernel at ~1.5 TB/s of output).
__device__ __forceinline__ void store_rows(float* __restrict__ dst, long long ldo, const uint32_t (&r)[32], float bv, bool cok, int nr) {
  if (nr == 32) {
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      if (cok) __stcs(dst, __uint_as_float(r[i]) + bv);
      dst += ldo;
    }
  } else {
#pragma unroll 1
    for (int i = 0; i < nr; ++i) {
      // r[] must stay in registers: select by a constant-index chain
      float v = 0.f;
#pragma unroll
      for (int k = 0; k < 32; ++k) v = (k == i) ? __uint_as_float(r[k]) : v;
      if (cok) __stcs(dst, v + bv);
      dst += ldo;
    }
  }
}

struct ScoreArgs {
  const float* bias;     // [n_cols]
  float* out;            // [n_rows, ldo]
  long long ldo;
  int n_cols;            // catalogue width N
  int n_rows;            // batch rows B
  int num_k;             // hp / 32
  int n_mtiles;          // ceil(N / 128)
  int n_chunks;          // ceil(B / NB)
};

// ============================================================================================
// CTA pairs (tcgen05 cta_group::2, thread-block cluster of 2): the two SMs of a
// pair compute one 256-column x NB-row tile. Each CTA loads its own 128 catalogue columns of A
// and HALF of the batch-row operand B; the pair's tensor cores read both halves, so the operand
// bytes per MMA drop from 48 KB to 32 KB per SM and k-block - one CTA per tile is bound by
// exactly that feed (profiles/r01_ncu_full_k_score_tc_v1.txt). Protocol:
//   * TMA of both CTAs completes on the LEADER's (cluster rank 0) full barrier;
//   * the leader's elected thread issues the MMAs for the pair and commits with a multicast
//     arrive, which frees the smem stage in both CTAs and hands the accumulator to both epilogues;
//   * each CTA drains its own 128 TMEM lanes; all 8 epilogue warps of the pair arrive on the
//     leader's accumulator-empty barrier (the peer's through a cluster-mapped address).
// ============================================================================================
template <int NB>
struct ScoreCfg2 {
  static_assert(NB == 64 || NB == 128 || NB == 256, "batch chunk must be 64, 128 or 256 rows");
  static constexpr int A_BYTES = TILE_M * BLOCK_K * 4;
  static constexpr int B_BYTES = (NB / 2) * BLOCK_K * 4;                 // this CTA's half of the batch rows
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = (200 * 1024 / STAGE_BYTES) > 8 ? 8 : (200 * 1024 / STAGE_BYTES);
  static constexpr int BAR_BYTES = 256;
  static constexpr int SMEM = STAGES * STAGE_BYTES + BAR_BYTES + 1024;
  static constexpr int TMEM_COLS = 2 * NB;
  // M = 256 over the pair, N = NB
  static constexpr uint32_t IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(NB >> 3) << 17) |
                                    ((uint32_t)((2 * TILE_M) >> 4) << 24);
};

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same variable in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_rank(const void* p, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(p)), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tma_load_2d_pair(void* dst, const CUtensorMap* map, uint32_t leader_bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(leader_bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma_tf32_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrives on the barrier at this shared-memory offset in BOTH CTAs of the pair once the MMAs issued so far are done.
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}

template <int NB>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NTHREADS, 1)
k_score_tc2(const __grid_constant__ CUtensorMap map_w, const __grid_constant__ CUtensorMap map_h, ScoreArgs a) {
  using C = ScoreCfg2<NB>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::STAGES * C::STAGE_BYTES);
  uint64_t* full = bars;                      // [STAGES] used in the leader: TMA of both CTAs -> MMA
  uint64_t* empty = bars + C::STAGES;         // [STAGES] in each CTA: MMA -> this CTA's TMA
  uint64_t* tfull = bars + 2 * C::STAGES;     // [2] in each CTA: MMA -> this CTA's epilogue
  uint64_t* tempty = tfull + 2;               // [2] used in the leader: both epilogues -> MMA
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(tempty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  const int n_ptiles = (a.n_mtiles + 1) / 2;              // 256-column tiles
  const int total = n_ptiles * a.n_chunks;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < C::STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&tfull[s], 1); mbar_init(&tempty[s], 2 * EPI_WARPS); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_holder)), "r"((uint32_t)C::TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  cluster_sync_all();                                      // both CTAs' barriers exist before anything arrives remotely
  tcgen05_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_holder);

  if (warp == 0) {
    int stage = 0; uint32_t phase = 0;
    for (int t = pair; t < total; t += n_pairs) {
      const int m = t / a.n_chunks, n = t - m * a.n_chunks;
      for (int k = 0; k < a.num_k; ++k) {
        mbar_wait(&empty[stage], phase ^ 1u);
        if (elect_one()) {
          uint8_t* sa = smem + stage * C::STAGE_BYTES;
          const uint32_t lbar = map_to_rank(&full[stage], 0);
          if (leader) mbar_expect_tx(&full[stage], 2u * (uint32_t)C::STAGE_BYTES);   // this CTA's boxes + the peer's
          tma_load_2d_pair(sa, &map_w, lbar, k * BLOCK_K, (2 * m + (int)rank) * TILE_M);
          tma_load_2d_pair(sa + C::A_BYTES, &map_h, lbar, k * BLOCK_K, n * NB + (int)rank * (NB / 2));
        }
        __syncwarp();
        if (++stage == C::STAGES) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    if (leader) {
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      for (int t = pair; t < total; t += n_pairs) {
        mbar_wait(&tempty[acc], acc_phase ^ 1u);
        tcgen05_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * NB);
        for (int k = 0; k < a.num_k; ++k) {
          mbar_wait(&full[stage], phase);
          tcgen05_fence_after();
          if (elect_one()) {
            const uint8_t* sa = smem + stage * C::STAGE_BYTES;
            const uint64_t da = make_desc(sa), db = make_desc(sa + C::A_BYTES);
#pragma unroll
            for (int kk = 0; kk < BLOCK_K / UMMA_K; ++kk)
              umma_tf32_pair(d_tmem, da + (uint64_t)(kk * 2), db + (uint64_t)(kk * 2), C::IDESC, (uint32_t)((k | kk) != 0));
            umma_commit_pair(&empty[stage]);
            if (k == a.num_k - 1) umma_commit_pair(&tfull[acc]);
          }
          __syncwarp();
          if (++stage == C::STAGES) { stage = 0; phase ^= 1u; }
        }
        acc ^= 1; if (acc == 0) acc_phase ^= 1u;
      }
    }
  } else {
    const int q = warp & 3;
    int acc = 0; uint32_t acc_phase = 0;
    for (int t = pair; t < total; t += n_pairs) {
      const int m = t / a.n_chunks, n = t - m * a.n_chunks;
      mbar_wait(&tfull[acc], acc_phase);
      tcgen05_fence_after();
      const int c = (2 * m + (int)rank) * TILE_M + q * 32 + lane;
      const bool cok = c < a.n_cols;
      const float bv = cok ? __ldg(a.bias + c) : 0.f;
      const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * NB);
#pragma unroll 1
      for (int j = (warp - 2) >> 2; j < NB / 32; j += EPI_WARPS / 4) {
        const int row0 = n * NB + j * 32;
        if (row0 >= a.n_rows) break;          // warp-uniform
        uint32_t r[32];
        tmem_ld32(tbase + (uint32_t)(j * 32), r);
        tmem_wait_ld();
        store_rows(a.out + (long long)row0 * a.ldo + c, a.ldo, r, bv, cok, min(32, a.n_rows - row0));
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(map_to_rank(&tempty[acc], 0));
      acc ^= 1; if (acc == 0) acc_phase ^= 1u;
    }
  }
  tcgen05_fence_before();
  cluster_sync_all();                                      // the peer may still be reading this CTA's operands / signalling its barriers
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)C::TMEM_COLS) : "memory");
  }
}

// ---- host side: tensor maps through the driver entry point (libcuda is not linked) -----------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

// K-major fp32 matrix [rows, hp] (row stride hp floats) cut into [box_rows x 32] boxes, 128-byte swizzle.
// The copy engine rounds fp32 to tf32 on the way in (the MMA alone would truncate).
inline int make_map(CUtensorMap* map, const float* base, int hp, long long rows, int box_rows) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(OCF_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
  cuuint64_t gdim[2] = {(cuuint64_t)hp, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)hp * sizeof(float)};
  cuuint32_t box[2] = {(cuuint32_t)BLOCK_K, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_TFLOAT32, 2,
                  const_cast<float*>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(OCF_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r));
  return OCF_OK;
}

template <int NB>
inline int launch_score_pair_nb(const CUtensorMap& mw, const CUtensorMap& mh, const ScoreArgs& a, int sm_count, cudaStream_t st) {
  using C = ScoreCfg2<NB>;
  static bool attr_set = false;
  if (!attr_set) {
    OCF_CUDA(cudaFuncSetAttribute(k_score_tc2<NB>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM));
    attr_set = true;
  }
  const int total = ((a.n_mtiles + 1) / 2) * a.n_chunks;
  const int pairs = total < sm_count / 2 ? total : sm_count / 2;
  k_score_tc2<NB><<<2 * pairs, NTHREADS, C::SMEM, st>>>(mw, mh, a);
  OCF_LAUNCHED();
  return OCF_OK;
}

inline int chunk_rows(int n_rows) { return n_rows <= 64 ? 64 : (n_rows <= 128 ? 128 : 256); }

}  // namespace tc
}  // namespace ocf
