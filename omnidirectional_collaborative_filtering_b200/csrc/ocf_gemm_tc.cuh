// Dense contractions of the training step on the 5th-generation tensor cores (tcgen05 + TMEM + TMA), sm_100a only:
// the hidden [H1, H2] layers of a deep model (model.py:64-71) forward, backward and weight-gradient + optimizer,
// and - when a batch is a true dense contraction (Jester-like stores, DESIGN.md section 4) - the encoder and decoder
// products themselves.
//
// One kernel, three operand arrangements. The accumulator tile is always [128 TMEM lanes x NB columns] with the
// CONTIGUOUS dimension of the output array along the lanes, so every epilogue store / read-modify-write is a
// 128-byte coalesced row per warp and register index:
//
//   forward   D[n, b] = sum_k W[k, n] h[b, k]      A = W   (MN-major: n contiguous)   B = h   (K-major)   -> a[b, n]
//   backward  D[k, b] = sum_n W[k, n] dz[b, n]     A = W   (K-major)                  B = dz  (K-major)   -> dz'[b, k]
//   gradient  D[n, k] = sum_b dz[b, n] h[b, k]     A = dz  (MN-major)                 B = h   (MN-major)  -> W[k, n] updated in place
//
// fp32 in, fp32-grade out: the tensor cores take tf32 operands (10 mantissa bits), which is too coarse for a
// gradient that Adagrad normalises to +-lr, so every operand tile is split in shared memory into hi = tf32(x) and
// lo = x - hi (exact) and the product is accumulated as hi*hi + hi*lo + lo*hi in fp32 TMEM ("3xTF32"; the dropped
// lo*lo term is 2^-22 relative). The contractions are tiny (<= 0.3 GFLOP): tensor time is irrelevant, what matters is
// that a [128 x 128 x 1024] product is spread over 32 SMs and leaves in ~3 us instead of a 64x64 SIMT tiling plus a
// split-K reduction kernel.
//
// Split-K without a second kernel and without float atomics: the CTAs of a thread-block cluster (<= 8, along the
// contraction) each contract their K range into TMEM, park the accumulator tile in their own shared memory, and after
// a cluster barrier every CTA sums a 1/S slice of the tile's columns over all ranks IN RANK ORDER through distributed
// shared memory (ld.shared::cluster) and runs the epilogue on it. Bit-reproducible.
//
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = TMEM owner + MMA issuer, warps 2..9 = operand splitters
// during the main loop, then epilogue (two warps per TMEM lane quarter, alternating column groups).
#pragma once

#include <cuda.h>

#include "ocf_common.cuh"
#include "ocf_kernels.cuh"
#include "ocf_score_tc.cuh"

namespace ocf {
namespace gtc {

using tc::smem_u32;

constexpr int GM = 128;            // accumulator rows = TMEM lanes = UMMA M
constexpr int NB = 128;            // accumulator columns per tile = UMMA N
constexpr int BK = 32;             // contraction elements per stage (one 128-byte swizzle row)
constexpr int EPI_WARPS = 8;         // two per TMEM lane quarter; also the operand splitters of the main loop
constexpr int NTHREADS = 64 + 32 * EPI_WARPS;
constexpr int TILE_BYTES = GM * BK * 4;              // 16 KB: one operand tile of a stage (A and B are both 128 x 32)
constexpr int STAGE_BYTES = 4 * TILE_BYTES;          // A hi | B hi | A lo | B lo
constexpr int STAGES = 3;
constexpr int PART_BYTES = NB * GM * 4;              // 64 KB accumulator tile parked for the cluster reduction (aliases the stage ring)
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 256 + 1024;
constexpr int MAX_SPLIT = 8;

enum { GEPI_FWD = 0, GEPI_DZ = 1, GEPI_UPDATE = 2, GEPI_STORE = 3, GEPI_RAW = 4 };

struct GemmTcArgs {
  int kind;
  int a_mn, b_mn;        // operand is MN-major (its tensor map is {MN inner, K rows}, loaded as 32 x 32 boxes)
  int k_blocks;          // 32-element blocks of the contraction each CTA handles
  int split;             // CTAs of a cluster along the contraction (gridDim.z)
  int m_valid;           // rows of the output that exist (the rest of the last tile is skipped)
  int n_valid;           // columns of the output that exist (batch rows for FWD / DZ, fan-in rows for UPDATE)
  int terms;             // 3 (or 0): hi*hi + hi*lo + lo*hi; 1: plain tf32 (diagnostic)
  float* C; int ldc;     // DZ: dz' [b, ldc]; UPDATE / STORE: W [k, ldc]; RAW: out [col, ldc]
  const float* aux0;     // DZ: activations a [b, ldc]
  const float* aux1;     // DZ: dropout scale [b, ldc] or null
  float* s1; float* s2;  // UPDATE: optimizer state, laid out like C
  int act;
  OptDev opt;
  ActArgs actargs;       // FWD: bias + activation + dropout of the layer (a_out / h_out / dscale are [b, hp4 * 4])
  unsigned long long* dbg;   // diagnostic (scripts/gemm_tc_bench.py): 8 %globaltimer stamps of CTA (0,0,0), else null
};

__device__ __forceinline__ void stamp(const GemmTcArgs& g, int slot) {
  if (g.dbg != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && threadIdx.x == 64) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    g.dbg[slot] = t;
  }
}

// instruction descriptor (kind::tf32): D = f32, A = B = tf32, M = 128, N = NB; bits 15 / 16 = A / B is MN-major
__host__ __device__ constexpr uint32_t idesc_of(bool a_mn, bool b_mn) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
         ((uint32_t)(NB >> 3) << 17) | ((uint32_t)(GM >> 4) << 24);
}

// Shared-memory matrix descriptors (version 1 = Blackwell).
//   K-major tile [128 rows x 32 tf32], layout type 2 (SWIZZLE_128B, 16-byte chunks): rows 128 bytes apart, 8-row
//     groups 1024 bytes apart (SBO); one MMA (K = 8) advances 32 bytes inside the swizzle row.
//   MN-major tile: for 32-bit operands the tensor core reads MN-major data only in layout type 1
//     (SWIZZLE_128B_BASE32B: 32-byte chunks swizzled over 4 rows; TMA writes it as SWIZZLE_128B_ATOM_32B). The tile
//     is four [32 k x 32 mn] boxes of 4 KB: inside a box a k-row is 128 bytes (32 mn elements), 4 k-rows form the
//     512-byte swizzle atom (SBO = 512 between k-groups), the next 32 mn elements are the next box (LBO = 4096);
//     one MMA (K = 8) spans two atoms and advances 1024 bytes.
__device__ __forceinline__ uint64_t desc_k_major(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
__device__ __forceinline__ uint64_t desc_mn_major(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)(4096 >> 4) << 16;
  d |= (uint64_t)(512 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)1 << 61;
  return d;
}

__device__ __forceinline__ float ld_dsmem(uint32_t cluster_addr) {
  float v;
  asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(cluster_addr) : "memory");
  return v;
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Epilogue of EB consecutive output columns of one row (m = index along the lanes, contiguous in memory). Every
// global load of the batch is issued before the first dependent instruction: one column at a time the epilogue was a
// chain of L2 round trips (load W / state -> update -> store, 32..64 times per thread) and cost 10x the contraction.
constexpr int EB = 8;

struct EpiRegs {            // per-thread constants of the epilogue, read once
  float lr; float bias; uint32_t drop_step; uint2 drop_key; uint32_t drop_thresh; float drop_inv;
};

struct EpiPre { float a[EB], b[EB], c[EB]; };      // what the batch's epilogue reads from global memory

// issued before the distributed-shared-memory reduction of the batch, so both latencies overlap
__device__ __forceinline__ void epi_prefetch(const GemmTcArgs& g, int m, int c_first, int n_ok, EpiPre& p) {
  if (g.kind == GEPI_DZ) {
#pragma unroll
    for (int j = 0; j < EB; ++j) {
      const size_t idx = (size_t)(c_first + j) * g.ldc + m;
      p.a[j] = j < n_ok ? __ldcg(g.aux0 + idx) : 0.f;
      p.b[j] = (j < n_ok && g.aux1 != nullptr) ? __ldcg(g.aux1 + idx) : 1.f;
    }
  } else if (g.kind == GEPI_UPDATE) {
#pragma unroll
    for (int j = 0; j < EB; ++j) {
      const size_t idx = (size_t)(c_first + j) * g.ldc + m;
      p.a[j] = j < n_ok ? __ldcg(g.C + idx) : 0.f;
      p.b[j] = (j < n_ok && g.s1 != nullptr) ? __ldcg(g.s1 + idx) : 0.f;
      p.c[j] = (j < n_ok && g.s2 != nullptr) ? __ldcg(g.s2 + idx) : 0.f;
    }
  }
}

__device__ __forceinline__ void epi_apply(const GemmTcArgs& g, const EpiRegs& e, int m, int c_first, int n_ok, const float (&v)[EB], EpiPre& p) {
  switch (g.kind) {
    case GEPI_FWD: {            // m = hidden unit n, columns = batch rows b
      const ActArgs& a = g.actargs;
#pragma unroll
      for (int j = 0; j < EB; ++j) {
        if (j >= n_ok) break;
        const int c = c_first + j;
        const size_t idx = (size_t)c * (a.hp4 * 4) + m;
        float z = v[j] + e.bias;
        z = (m < a.H) ? act_fwd(a.act, z) : 0.f;
        reinterpret_cast<float*>(a.a_out)[idx] = z;
        if (a.dscale != nullptr) {
          const uint4 r = philox4x32_10(make_uint4((uint32_t)(m >> 2), (uint32_t)(c + a.row0), a.layer, e.drop_step), e.drop_key);
          const uint32_t rr = (m & 3) == 0 ? r.x : ((m & 3) == 1 ? r.y : ((m & 3) == 2 ? r.z : r.w));
          const float sc = ((rr >> 8) >= e.drop_thresh) ? e.drop_inv : 0.f;
          reinterpret_cast<float*>(a.dscale)[idx] = sc;
          z *= sc;
        }
        reinterpret_cast<float*>(a.h_out)[idx] = z;
      }
    } break;
    case GEPI_DZ:               // m = unit k of the layer below, columns = batch rows b
#pragma unroll
      for (int j = 0; j < EB; ++j)
        if (j < n_ok) g.C[(size_t)(c_first + j) * g.ldc + m] = v[j] * p.b[j] * act_bwd(g.act, p.a[j]);
      break;
    case GEPI_UPDATE:           // m = fan-out n, columns = fan-in k: W[k, n]
#pragma unroll
      for (int j = 0; j < EB; ++j) {
        if (j >= n_ok) break;
        const size_t idx = (size_t)(c_first + j) * g.ldc + m;
        opt_apply(g.opt, e.lr, v[j], p.a[j], p.b[j], p.c[j]);
        g.C[idx] = p.a[j];
        if (g.s1) g.s1[idx] = p.b[j];
        if (g.s2) g.s2[idx] = p.c[j];
      }
      break;
    default:                    // STORE / RAW: out[c, m]
#pragma unroll
      for (int j = 0; j < EB; ++j)
        if (j < n_ok) g.C[(size_t)(c_first + j) * g.ldc + m] = v[j];
      break;
  }
}

__global__ void __launch_bounds__(NTHREADS, 1)
k_gemm_tc(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, GemmTcArgs g) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
  uint64_t* full = bars;                  // [STAGES] TMA -> splitter
  uint64_t* ready = bars + STAGES;        // [STAGES] splitter -> MMA
  uint64_t* empty = bars + 2 * STAGES;    // [STAGES] MMA -> TMA
  uint64_t* tfull = bars + 3 * STAGES;    // [1] MMA -> epilogue
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(tfull + 1);

  pdl_trigger();
  stamp(g, 0);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.x * GM;             // first output row (lane dimension) of the tile
  const int c0 = blockIdx.y * NB;             // first output column
  const int kb0 = blockIdx.z * g.k_blocks;    // first contraction block of this CTA
  const uint32_t rank = g.split > 1 ? tc::cluster_ctarank() : 0u;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) { tc::mbar_init(&full[s], 1); tc::mbar_init(&ready[s], EPI_WARPS); tc::mbar_init(&empty[s], 1); }
    tc::mbar_init(tfull, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_holder)), "r"((uint32_t)NB) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc::tcgen05_fence_before();
  __syncthreads();
  tc::tcgen05_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_holder);
  pdl_wait();                                 // barriers and TMEM are set up while the previous kernel drains
  stamp(g, 1);

  if (warp == 0) {
    // ---- TMA producer: raw fp32 tiles into the hi halves of the stage ------------------------------------
    int stage = 0; uint32_t phase = 0;
    for (int k = 0; k < g.k_blocks; ++k) {
      tc::mbar_wait(&empty[stage], phase ^ 1u);
      if (tc::elect_one()) {
        uint8_t* sa = smem + stage * STAGE_BYTES;
        uint8_t* sb = sa + TILE_BYTES;
        const int kk = (kb0 + k) * BK;
        tc::mbar_expect_tx(&full[stage], 2u * TILE_BYTES);
        if (g.a_mn) { for (int q = 0; q < 4; ++q) tc::tma_load_2d(sa + q * 4096, &map_a, &full[stage], m0 + q * 32, kk); }
        else tc::tma_load_2d(sa, &map_a, &full[stage], kk, m0);
        if (g.b_mn) { for (int q = 0; q < 4; ++q) tc::tma_load_2d(sb + q * 4096, &map_b, &full[stage], c0 + q * 32, kk); }
        else tc::tma_load_2d(sb, &map_b, &full[stage], kk, c0);
      }
      __syncwarp();
      if (++stage == STAGES) { stage = 0; phase ^= 1u; }
    }
  } else if (warp == 1) {
    // ---- MMA issuer ------------------------------------------------------------------------------------
    const uint32_t idesc = idesc_of(g.a_mn != 0, g.b_mn != 0);
    const uint64_t step_a = g.a_mn ? (1024 >> 4) : (32 >> 4), step_b = g.b_mn ? (1024 >> 4) : (32 >> 4);
    int stage = 0; uint32_t phase = 0;
    for (int k = 0; k < g.k_blocks; ++k) {
      tc::mbar_wait(&ready[stage], phase);
      tc::tcgen05_fence_after();
      if (tc::elect_one()) {
        const uint32_t sa = smem_u32(smem + stage * STAGE_BYTES);
        const uint64_t ah = g.a_mn ? desc_mn_major(sa) : desc_k_major(sa);
        const uint64_t bh = g.b_mn ? desc_mn_major(sa + TILE_BYTES) : desc_k_major(sa + TILE_BYTES);
        const uint64_t al = g.a_mn ? desc_mn_major(sa + 2 * TILE_BYTES) : desc_k_major(sa + 2 * TILE_BYTES);
        const uint64_t bl = g.b_mn ? desc_mn_major(sa + 3 * TILE_BYTES) : desc_k_major(sa + 3 * TILE_BYTES);
#pragma unroll
        for (int kk = 0; kk < BK / 8; ++kk) {
          const uint64_t oa = (uint64_t)kk * step_a, ob = (uint64_t)kk * step_b;
          if (g.terms == 3) {
            // small terms first, so they are not added to an already large accumulator one at a time
            tc::umma_tf32(tmem_base, al + oa, bh + ob, idesc, (uint32_t)((k | kk) != 0));
            tc::umma_tf32(tmem_base, ah + oa, bl + ob, idesc, 1u);
            tc::umma_tf32(tmem_base, ah + oa, bh + ob, idesc, 1u);
          } else {
            tc::umma_tf32(tmem_base, ah + oa, bh + ob, idesc, (uint32_t)((k | kk) != 0));
          }
        }
        tc::umma_commit(&empty[stage]);
        if (k == g.k_blocks - 1) tc::umma_commit(tfull);
      }
      __syncwarp();
      if (++stage == STAGES) { stage = 0; phase ^= 1u; }
    }
  } else {
    // ---- operand splitter: x -> hi = tf32(x) (round to nearest, in place), lo = x - hi (exact) ----------
    const int t = threadIdx.x - 64;        // 0..255
    int stage = 0; uint32_t phase = 0;
    for (int k = 0; k < g.k_blocks; ++k) {
      tc::mbar_wait(&full[stage], phase);
      if (k == 0) stamp(g, 2);
      float4* hi = reinterpret_cast<float4*>(smem + stage * STAGE_BYTES);
      float4* lo = hi + 2 * TILE_BYTES / 16;
#pragma unroll 4
      for (int i = t; i < 2 * TILE_BYTES / 16; i += 32 * EPI_WARPS) {
        const float4 x = hi[i];
        float4 h, l;
        h.x = __uint_as_float((__float_as_uint(x.x) + 0x1000u) & 0xFFFFE000u); l.x = x.x - h.x;
        h.y = __uint_as_float((__float_as_uint(x.y) + 0x1000u) & 0xFFFFE000u); l.y = x.y - h.y;
        h.z = __uint_as_float((__float_as_uint(x.z) + 0x1000u) & 0xFFFFE000u); l.z = x.z - h.z;
        h.w = __uint_as_float((__float_as_uint(x.w) + 0x1000u) & 0xFFFFE000u); l.w = x.w - h.w;
        hi[i] = h;
        lo[i] = l;
      }
      fence_async_smem();                  // generic-proxy writes -> visible to the tensor core's async-proxy reads
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&ready[stage]);
      if (++stage == STAGES) { stage = 0; phase ^= 1u; }
    }
  }

  // ---- epilogue -------------------------------------------------------------------------------------------
  const int q = warp & 3;                      // TMEM lane quarter of an epilogue warp
  const int half = warp >= 6 ? 1 : 0;          // the two warps of a quarter alternate column groups
  const int ml = q * 32 + lane;                // row of the tile this thread owns
  const int m = m0 + ml;
  EpiRegs e{};
  if (warp >= 2) {
    if (g.kind == GEPI_UPDATE) e.lr = g.opt.st->lr;
    if (g.kind == GEPI_FWD) e.bias = m < g.m_valid ? reinterpret_cast<const float*>(g.actargs.bias)[m] : 0.f;
    if (g.kind == GEPI_FWD && g.actargs.dscale != nullptr) {
      e.drop_step = g.actargs.st->step; e.drop_key = make_uint2(g.actargs.st->seed_lo, g.actargs.st->seed_hi);
      e.drop_thresh = (uint32_t)floor((double)g.actargs.p_drop * 16777216.0);
      e.drop_inv = 1.0f / (1.0f - g.actargs.p_drop);
    }
    tc::mbar_wait(tfull, 0);
    tc::tcgen05_fence_after();
    stamp(g, 3);
  }
  if (g.split == 1) {
    if (warp >= 2) {
      const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
      for (int j = half; j < NB / 32; j += 2) {
        if (c0 + j * 32 >= g.n_valid) break;
        uint32_t r[32];
        tc::tmem_ld32(tbase + (uint32_t)(j * 32), r);
        tc::tmem_wait_ld();
#pragma unroll
        for (int i0 = 0; i0 < 32; i0 += EB) {
          const int cf = c0 + j * 32 + i0;
          if (m < g.m_valid && cf < g.n_valid) {
            const int n_ok = min(EB, g.n_valid - cf);
            EpiPre pre;
            epi_prefetch(g, m, cf, n_ok, pre);
            float v[EB];
#pragma unroll
            for (int i = 0; i < EB; ++i) v[i] = __uint_as_float(r[i0 + i]);
            epi_apply(g, e, m, cf, n_ok, v, pre);
          }
        }
      }
    }
  } else {
    // park the tile: part[col][row], rows contiguous (conflict-free stores, coalesced remote loads)
    float* part = reinterpret_cast<float*>(smem);
    if (warp >= 2) {
      const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
      for (int j = half; j < NB / 32; j += 2) {
        uint32_t r[32];
        tc::tmem_ld32(tbase + (uint32_t)(j * 32), r);
        tc::tmem_wait_ld();
#pragma unroll
        for (int i = 0; i < 32; ++i) part[(j * 32 + i) * GM + ml] = __uint_as_float(r[i]);
      }
    }
    tc::cluster_sync_all();
    stamp(g, 4);
    if (warp >= 2) {
      const int cps = NB / g.split;              // columns this CTA reduces and finishes (16, 32 or 64: multiples of 2 * EB)
      uint32_t base[MAX_SPLIT];
#pragma unroll
      for (int r = 0; r < MAX_SPLIT; ++r) base[r] = tc::map_to_rank(part, (uint32_t)(r < g.split ? r : 0));
#pragma unroll 1
      for (int i0 = half * EB; i0 < cps; i0 += 2 * EB) {
        const int cl = (int)rank * cps + i0;
        const int cf = c0 + cl;
        if (cf >= g.n_valid) break;
        const int n_ok = min(EB, g.n_valid - cf);
        EpiPre pre;
        if (m < g.m_valid) epi_prefetch(g, m, cf, n_ok, pre);
        const uint32_t off = (uint32_t)((cl * GM + ml) * 4);
        // every rank's values of the batch first (one round trip over the cluster), then the sums in rank order
        float u[MAX_SPLIT][EB];
#pragma unroll
        for (int r = 0; r < MAX_SPLIT; ++r) {
          if (r < g.split) {
#pragma unroll
            for (int i = 0; i < EB; ++i) u[r][i] = ld_dsmem(base[r] + off + (uint32_t)(i * GM * 4));
          }
        }
        float v[EB];
#pragma unroll
        for (int i = 0; i < EB; ++i) v[i] = u[0][i];
#pragma unroll
        for (int r = 1; r < MAX_SPLIT; ++r) {
          if (r < g.split) {
#pragma unroll
            for (int i = 0; i < EB; ++i) v[i] += u[r][i];
          }
        }
        if (m < g.m_valid) epi_apply(g, e, m, cf, n_ok, v, pre);
      }
    }
    stamp(g, 5);
    tc::cluster_sync_all();                      // nobody leaves while a peer still reads its tile
  }
  stamp(g, 6);
  tc::tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc::tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)NB) : "memory");
  }
  stamp(g, 7);
}

// ---- host side -----------------------------------------------------------------------------------------------
// K-major operand: array [rows, ld] contracted along its contiguous dimension; boxes [128 rows x 32].
inline int make_map_k(CUtensorMap* map, const float* base, long long k_len, long long ld, long long rows) {
  tc::EncodeTiledFn fn = tc::encode_fn();
  if (!fn) return fail(OCF_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
  cuuint64_t gdim[2] = {(cuuint64_t)k_len, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)ld * sizeof(float)};
  cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)GM};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(OCF_ERR_CUDA, "cuTensorMapEncodeTiled (K-major) failed with CUresult " + std::to_string((int)r));
  return OCF_OK;
}
// MN-major operand: array [k_rows, ld] contracted along its rows; boxes [32 k-rows x 32 contiguous elements].
// Rows beyond k_rows and elements beyond mn_len read as zero (they must: they are part of the contraction).
inline int make_map_mn(CUtensorMap* map, const float* base, long long mn_len, long long ld, long long k_rows) {
  tc::EncodeTiledFn fn = tc::encode_fn();
  if (!fn) return fail(OCF_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
  cuuint64_t gdim[2] = {(cuuint64_t)mn_len, (cuuint64_t)k_rows};
  cuuint64_t gstride[1] = {(cuuint64_t)ld * sizeof(float)};
  cuuint32_t box[2] = {32u, (cuuint32_t)BK};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(OCF_ERR_CUDA, "cuTensorMapEncodeTiled (MN-major) failed with CUresult " + std::to_string((int)r));
  return OCF_OK;
}

// Contraction split: cluster ranks (power of two, <= 8) share out the 32-element blocks until the launch has ~128
// CTAs: the epilogue (read-modify-write of the weights, or the activation stores) is then spread as widely as the
// contraction, and it is the longer part.
inline int pick_split(int total_k_blocks, int tiles) {
  int s = 1;
  while (s < MAX_SPLIT && total_k_blocks % (2 * s) == 0 && tiles * s < 128) s *= 2;
  return s;
}

// D[m_len, n_len] over a contraction of k_len elements (a multiple of 32 after zero fill).
inline int launch(const CUtensorMap& ma, const CUtensorMap& mb, GemmTcArgs g, int m_len, int n_len, int k_len, cudaStream_t st,
                  int want_split = 0, bool pdl = false) {
  static bool attr_set = false;
  if (!attr_set) {
    OCF_CUDA(cudaFuncSetAttribute(k_gemm_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    attr_set = true;
  }
  const int mt = (m_len + GM - 1) / GM, nt = (n_len + NB - 1) / NB;
  const int kb = (k_len + BK - 1) / BK;
  int split = pick_split(kb, mt * nt);
  if (want_split >= 1 && want_split <= MAX_SPLIT) { split = want_split; while (kb % split) split /= 2; }
  g.split = split;
  g.k_blocks = kb / split;
  g.m_valid = m_len; g.n_valid = n_len;
  if (g.terms == 0) g.terms = 3;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)mt, (unsigned)nt, (unsigned)split);
  cfg.blockDim = dim3(NTHREADS, 1, 1);
  cfg.dynamicSmemBytes = SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute at[2];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 1; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = (unsigned)split;
  at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = pdl ? 2 : 1;
  OCF_CUDA(cudaLaunchKernelEx(&cfg, k_gemm_tc, ma, mb, g));
  OCF_LAUNCHED();
  return OCF_OK;
}

}  // namespace gtc
}  // namespace ocf
