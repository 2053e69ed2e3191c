// Grouped weight-gradient + Adam kernel: EVERY linear layer of EVERY ensemble member in ONE persistent launch at the
// end of the backward pass (reference: the autograd weight gradients of src/blocks.py's Linear layers followed by
// torch.optim.Adam.step, src/DGMMixin.py:121-123).
//
// Why one deferred launch.  Round 1 ran one fused dW+Adam GEMM per layer inside the backward chain: 11 launches,
// 51 % of the critical path, each a persistent kernel that owns all SMs while the latency-bound kernels of the other
// branch wait.  The weight gradients are needed by nothing but the optimizer, and all their inputs (layer inputs and
// pre-activation gradients, chunk8 buffers) stay alive until the end of the step, so the whole optimizer traffic
// (24 B/parameter) becomes one HBM stream with no tails between layers; the dX chain in front of it is then made of
// small kernels only.
//
// Why TMA for the optimizer state.  The per-thread epilogue of round 1 was bound by memory-level parallelism (resident
// warps x registers): 4.5-4.7 TB/s.  Here p, m, v of a tile are staged through shared memory by tensor loads
// ({128 k, 16 weight rows} boxes of the reference [out][in] tensors: 3 instructions per 24 KB stage) and written back by
// tensor stores together with the refreshed bf16 chunk8 shadow; the bytes in flight per SM no longer depend on the
// epilogue warps (tools/adam_tma_bench.cu: 5.4-5.7 TB/s = 87 % of the measured copy bandwidth).  Needs 16-byte aligned
// weight rows (plan.cu add_tensor) and 16-aligned stacking of two-head layers (a stage never straddles two tensors).
//
// Roles (20 warps, one CTA per SM, tiles strided over the grid):
//   warp 0   operand producer: TMA loads of the X^T / dY tiles (MN-major boxes) into a 2-stage ring
//   warp 1   state loader: TMA loads of p, m, v stages (runs ahead of the accumulator: next tile's state is prefetched)
//   warp 2   state storer: waits for a stage to be updated, TMA-stores p, m, v and the shadow, frees the stage
//   warp 3   tcgen05.mma issuer (M = 128 input features x BN weight rows, fp32 accumulators in TMEM, double-buffered)
//   warps 4-19  epilogue: lane = input feature (TMEM lane), 4 weight rows per warp and stage; Adam on shared memory
// D row k < kin is weight column k; k == kin (ones column of the layer input) is the bias gradient, staged per tile
// through a small shared array; k > kin are the one-hot class columns (weight column k - 1).
#pragma once

#include "gemm.cuh"

namespace drvae {

constexpr int DWA_MAX_LAYERS = 24;
constexpr int DWA_R = 16;          // weight rows per state stage
constexpr int DWA_NST = 4;         // state stages
constexpr int DWA_OPS = 2;         // operand stages
#ifndef DWA_EPI_WARPS
#define DWA_EPI_WARPS 8
#endif
constexpr int DWA_EW = DWA_EPI_WARPS;  // epilogue warps (8 or 16: warp w reads TMEM lane quarter w % 4; measured 16 -> 8: 0.402 -> 0.400 ms, fewer
                                       // instructions per parameter, profiles/r02_experiments.md)
constexpr int DWA_RPW = DWA_R * 4 / DWA_EW;  // weight rows of a stage per epilogue warp
static_assert(DWA_EW % 4 == 0 && DWA_RPW * DWA_EW == DWA_R * 4 && (DWA_RPW == 4 || DWA_RPW == 8), "epilogue geometry");
static_assert(DWA_EW * 32 >= 256, "the bias staging needs one epilogue thread per tile column");
constexpr int DWA_THREADS = (4 + DWA_EW) * 32;
// Register budget.  Compiled for two resident CTAs (80 registers) the kernel would leave half of the register file to
// the row kernels that run next to the early launch (plan.cu) — measured: the launch alone 0.394 -> 0.408 ms, the step
// with the early launch the same within noise (0.911-0.918 ms either way), the step without it 0.940 -> 0.951 ms.
#ifndef DWA_MIN_BLOCKS
#define DWA_MIN_BLOCKS 1
#endif
constexpr int DWA_OP_STAGE = GEMM_A_STAGE_BYTES + 256 * GEMM_BK * 2;  // 48 KB
constexpr int DWA_ARR = DWA_R * 128 * 4;                              // one array of a state stage
constexpr int DWA_SHB = DWA_R * 256;                                  // bf16 shadow of a stage: [16 chunks][R][8]
constexpr int DWA_ST_STAGE = 3 * DWA_ARR + DWA_SHB;                   // 28 KB
constexpr int DWA_BIAS_BYTES = 4 * 256 * 4;                           // b, m, v, flat offset for up to 256 weight rows
constexpr int DWA_SMEM = DWA_OPS * DWA_OP_STAGE + DWA_NST * DWA_ST_STAGE + DWA_BIAS_BYTES + 1024;

struct DwaMaps {  // per layer, global memory, 64-byte aligned
  CUtensorMap A, B;              // operand tiles: {64 rows, 16 chunks} of the layer input, {64 rows, BN/8 chunks} of dY
  CUtensorMap P[2], M[2], V[2];  // optimizer state of the (up to two stacked) weight tensors: {ld, rows, models}, box {128, R, 1}
  CUtensorMap S;                 // bf16 chunk8 shadow: box {R rows, 16 chunks, 1}
};

struct DwaLayer {
  int tile_begin, tile_end;
  int tiles_m, tiles_n, BN;
  int kin, kaug;            // true input features; kin + 1 (ones column) + class columns
  int cnt_which;            // counts[] entry with the contraction rows of this layer
  int a_row0;
  int ntens, rows_each, ilv_block, ilv_stride;
  int rcap;                 // shadow rows (tiles_n_fwd * BN_fwd): extent of the tables
  int skip_which;           // >= 0: counts[] entry; when it is zero the layer is not updated at all (PVAE p(z2|z1) with no
                            // pairs in the batch: the reference's gradient is None and torch.optim.Adam skips the tensor)
  long long tab_off;        // g_tab: [3][rcap] (weight row offsets, bias offsets, folded bias constants)
  long long drv_bias_off, drv_clsb_off;
  int drv_clsb_ld;
  int ld;                   // floats between rows of the weight tensors
  int w_off[2];             // flat offsets of the weight tensors
  long long sh_off;         // bf16 shadow of the layer inside the per-model shadow arena
};

struct DwaParams {
  int n_layers, n_models, total_tiles;
  int tile_begin, tile_end;  // tiles of this launch (the step may run the layers whose inputs are complete early, see plan.cu)
  const DwaLayer* layers;   // device
  const DwaMaps* maps;      // device
  const int* tabs;          // plan-wide gradient-epilogue tables
  const int* counts;
  int counts_stride;
  float *adam_p, *adam_m, *adam_v;
  long long state_ms;
  float* drv;
  long long drv_ms;
  bf16* shadow;             // shadow arena (direct-store variant)
  long long shadow_ms;
  const AdamHyper* adam;
  int adam_ms;              // bytes between the Adam scalars of consecutive models (0: shared)
  DebugWord* dbg;
  unsigned long long* trace;
  int trace_id;
  int debug_flags;            // measurement knob (DRVAE_B200_DWA_DEBUG): 1 = no operand loads / MMA (gradient = 0: NOT a valid step)
  unsigned long long* stats;  // optional [8] cycle counters of the roles' barrier waits (drvae_debug_dwa_stats)
};

__device__ __forceinline__ void tma_store_3d(const void* map, const void* src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"((unsigned long long)map),
               "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_wait_group_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_wait_group0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(DWA_EW * 32) : "memory"); }

// 32 lanes x 4 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, float (&v)[4]) {
  uint32_t r[4];
  __syncwarp();
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(taddr)
               : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 4; ++i) v[i] = __uint_as_float(r[i]);
}

enum { DWS_EPI_ACC = 0, DWS_EPI_STATE, DWS_LOADER_EMPTY, DWS_STORER_DONE, DWS_STORER_READ, DWS_PROD_EMPTY, DWS_MMA_FULL, DWS_CTA_TOTAL };
#define DWS_T0() const long long dws_t0 = (STATS && p.stats) ? clock64() : 0
#define DWS_ADD(acc) \
  if (STATS && p.stats) acc += clock64() - dws_t0

// issue / complete halves of a 4-column TMEM load (the load is in flight across a barrier wait)
__device__ __forceinline__ void tmem_ld4_issue(uint32_t taddr, uint32_t (&r)[4]) {
  __syncwarp();
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_ld4_wait(bool have, uint32_t (&r)[4], float (&v)[4]) {
  if (have) asm volatile("tcgen05.wait::ld.sync.aligned;" : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3])::"memory");
#pragma unroll
  for (int i = 0; i < 4; ++i) v[i] = have ? __uint_as_float(r[i]) : 0.f;
}

// RPW consecutive fp32 columns of 32 lanes, issue / wait halves
template <int N>
__device__ __forceinline__ void tmem_ldN_issue(uint32_t taddr, uint32_t (&r)[N]) {
  __syncwarp();
  if constexpr (N == 4) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(taddr)
                 : "memory");
  } else if constexpr (N == 8) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
  } else {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
  }
}
template <int N>
__device__ __forceinline__ void tmem_ldN_wait(bool have, uint32_t (&r)[N], float (&v)[N]) {
  if (have) asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < N; ++i) v[i] = have ? __uint_as_float(r[i]) : 0.f;
}

struct DwaTile {
  int layer, model, m0, n0, BN;
  int nkb, Kc;
  bool active;
};

__device__ __forceinline__ DwaTile dwa_tile(const DwaParams& p, const DwaLayer* L, int tile) {
  DwaTile t;
  int l = 0;
  while (l + 1 < p.n_layers && tile >= L[l].tile_end) ++l;
  t.layer = l;
  const DwaLayer& y = L[l];
  const int local = tile - y.tile_begin;
  const int per = y.tiles_m * y.tiles_n;
  t.model = local / per;
  const int mn = local - t.model * per;
  t.m0 = (mn % y.tiles_m) * GEMM_BM;  // consecutive tiles: consecutive 128-feature segments of the same weight rows
  t.n0 = (mn / y.tiles_m) * y.BN;
  t.BN = y.BN;
  const int rows = p.counts[(long long)t.model * p.counts_stride + y.cnt_which];
  t.Kc = (rows + 15) & ~15;
  t.nkb = (p.debug_flags & 1) ? 0 : (t.Kc + GEMM_BK - 1) / GEMM_BK;
  t.active = !(y.skip_which >= 0 && p.counts[(long long)t.model * p.counts_stride + y.skip_which] == 0);
  return t;
}

// weight tensor / row of the first shadow row of a stage; false: the stage holds no parameters
__device__ __forceinline__ bool dwa_stage_rows(const DwaLayer& y, int s0, int& which, int& n) {
  const int blk = s0 / y.ilv_stride, rem = s0 - blk * y.ilv_stride;
  which = rem / y.ilv_block;
  n = blk * y.ilv_block + (rem - which * y.ilv_block);
  return which < y.ntens && n < y.rows_each;
}

// STATS: instrumented instance (role wait counters, drvae_debug_dwa_stats); the production instance has none of it
template <bool STATS>
__global__ void __launch_bounds__(DWA_THREADS, DWA_MIN_BLOCKS) dwadam_kernel(const DwaParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t op_full[DWA_OPS], op_empty[DWA_OPS], acc_full[2], acc_empty[2];
  __shared__ __align__(8) uint64_t st_full[DWA_NST], st_done[DWA_NST], st_empty[DWA_NST];
  __shared__ uint32_t tmem_base_s;
  __shared__ DwaLayer L[DWA_MAX_LAYERS];

  // 1 KB alignment by pointer arithmetic on the __shared__ array itself: a round trip through an integer makes the
  // compiler lose the address space and emit generic LD/ST (seen in the SASS of the first version) instead of LDS/STS
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* op_ring = smem;
  uint8_t* st_ring = smem + DWA_OPS * DWA_OP_STAGE;
  float* bst = reinterpret_cast<float*>(st_ring + DWA_NST * DWA_ST_STAGE);  // [3][256] b, m, v
  int* bidx = reinterpret_cast<int*>(bst + 3 * 256);                         // [256] flat offset of b[n] or -1

  TraceScope trace_scope(p.trace, p.trace_id);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < DWA_OPS; ++s) {
      mbar_init(&op_full[s], 1);
      mbar_init(&op_empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&acc_full[a], 1);
      mbar_init(&acc_empty[a], DWA_EW);
    }
    for (int s = 0; s < DWA_NST; ++s) {
      mbar_init(&st_full[s], 1);
      mbar_init(&st_done[s], DWA_EW);
      mbar_init(&st_empty[s], 1);
    }
    mbar_fence_init();
  }
  if (warp == 3) {
    tmem_alloc(&tmem_base_s, 512);
    tmem_relinquish();
  }
  for (int i = threadIdx.x; i < p.n_layers * (int)(sizeof(DwaLayer) / 4); i += blockDim.x)
    reinterpret_cast<int*>(L)[i] = reinterpret_cast<const int*>(p.layers)[i];
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;
  long long w_a = 0, w_b = 0;  // wait-cycle counters of this thread's role (p.stats)
  const long long cta_t0 = (STATS && p.stats) ? clock64() : 0;

  if (warp == 0) {
    // ===================== operand producer =====================
    uint32_t it = 0;
    for (int tile = p.tile_begin + blockIdx.x; tile < p.tile_end; tile += gridDim.x) {
      const DwaTile t = dwa_tile(p, L, tile);
      if (!t.active) continue;
      const DwaLayer& y = L[t.layer];
      const DwaMaps* mp = p.maps + t.layer;
      const uint32_t tx = GEMM_A_STAGE_BYTES + t.BN * GEMM_BK * 2;
      for (int kb = 0; kb < t.nkb; ++kb, ++it) {
        const int s = it % DWA_OPS;
        {
          DWS_T0();
          mbar_wait_sleepy(&op_empty[s], ((it / DWA_OPS) & 1) ^ 1, p.dbg, 0xE1000000u | kb);
          DWS_ADD(w_a);
        }
        if (elect_one()) {
          uint8_t* As = op_ring + (size_t)s * DWA_OP_STAGE;
          mbar_arrive_expect_tx(&op_full[s], tx);
          tma_load_3d(As, &mp->A, (y.a_row0 + kb * GEMM_BK) * 2, t.m0 >> 3, t.model, &op_full[s]);
          tma_load_3d(As + GEMM_A_STAGE_BYTES, &mp->B, (kb * GEMM_BK) * 2, t.n0 >> 3, t.model, &op_full[s]);
        }
        __syncwarp();
      }
    }
  } else if (warp == 1) {
    // ===================== optimizer-state loader =====================
    uint32_t it = 0;
    for (int tile = p.tile_begin + blockIdx.x; tile < p.tile_end; tile += gridDim.x) {
      const DwaTile t = dwa_tile(p, L, tile);
      if (!t.active) continue;
      const DwaLayer& y = L[t.layer];
      const DwaMaps* mp = p.maps + t.layer;
      for (int sub = 0; sub < t.BN / DWA_R; ++sub, ++it) {
        const int s = it % DWA_NST;
        {
          DWS_T0();
          mbar_wait_sleepy(&st_empty[s], ((it / DWA_NST) & 1) ^ 1, p.dbg, 0xE2000000u | sub);
          DWS_ADD(w_a);
        }
        int which, n;
        const bool has = dwa_stage_rows(y, t.n0 + sub * DWA_R, which, n);
        if (elect_one()) {
          if (has) {
            uint8_t* st = st_ring + (size_t)s * DWA_ST_STAGE;
            mbar_arrive_expect_tx(&st_full[s], 3 * DWA_ARR);
            tma_load_3d(st, &mp->P[which], t.m0, n, t.model, &st_full[s]);
            tma_load_3d(st + DWA_ARR, &mp->M[which], t.m0, n, t.model, &st_full[s]);
            tma_load_3d(st + 2 * DWA_ARR, &mp->V[which], t.m0, n, t.model, &st_full[s]);
          } else {
            mbar_arrive(&st_full[s]);
          }
        }
        __syncwarp();
      }
    }
  } else if (warp == 2) {
    // ===================== optimizer-state storer =====================
    uint32_t it = 0;
    for (int tile = p.tile_begin + blockIdx.x; tile < p.tile_end; tile += gridDim.x) {
      const DwaTile t = dwa_tile(p, L, tile);
      if (!t.active) continue;
      const DwaLayer& y = L[t.layer];
      const DwaMaps* mp = p.maps + t.layer;
      for (int sub = 0; sub < t.BN / DWA_R; ++sub, ++it) {
        const int s = it % DWA_NST;
        {
          DWS_T0();
          mbar_wait_sleepy(&st_done[s], (it / DWA_NST) & 1, p.dbg, 0xE3000000u | sub);
          DWS_ADD(w_a);
        }
        int which, n;
        const int s0 = t.n0 + sub * DWA_R;
        const bool has = dwa_stage_rows(y, s0, which, n);
        if (elect_one()) {
          if (has) {
            uint8_t* st = st_ring + (size_t)s * DWA_ST_STAGE;
            tma_store_3d(&mp->P[which], st, t.m0, n, t.model);
            tma_store_3d(&mp->M[which], st + DWA_ARR, t.m0, n, t.model);
            tma_store_3d(&mp->V[which], st + 2 * DWA_ARR, t.m0, n, t.model);
            tma_store_3d(&mp->S, st + 3 * DWA_ARR, s0 * 2, t.m0 >> 3, t.model);
            tma_commit_group();
            DWS_T0();
            tma_wait_group_read0();  // the TMA unit has read this stage's shared memory
            DWS_ADD(w_b);
          }
          mbar_arrive(&st_empty[s]);
        }
        __syncwarp();
      }
    }
    if (elect_one()) tma_wait_group0();  // every write has landed before the CTA exits
    __syncwarp();
  } else if (warp == 3) {
    // ===================== UMMA issuer (weight-gradient mode: both operands MN-major) =====================
    if (elect_one()) {
      const uint64_t d0 = umma_smem_desc(0, 128, GEMM_BK * 16);
      const uint32_t hi = (uint32_t)(d0 >> 32), lo0 = (uint32_t)d0;
      const uint32_t smem0 = smem_u32(op_ring) >> 4, stage16 = (uint32_t)DWA_OP_STAGE >> 4;
      uint32_t it = 0, j = 0;
      for (int tile = p.tile_begin + blockIdx.x; tile < p.tile_end; tile += gridDim.x) {
        const DwaTile t = dwa_tile(p, L, tile);
        if (!t.active) continue;
        const uint32_t idesc = umma_idesc_bf16(t.BN, 1, 1);
        const uint32_t a = j & 1, aph = (j >> 1) & 1;
        mbar_wait_sleepy(&acc_empty[a], aph ^ 1, p.dbg, 0xB1000000u | tile);
        tc_fence_after();
        const uint32_t tacc = tmem_base + a * 256;
        for (int kb = 0; kb < t.nkb; ++kb, ++it) {
          const uint32_t s = it % DWA_OPS;
          {
            DWS_T0();
            mbar_wait_sleepy(&op_full[s], (it / DWA_OPS) & 1, p.dbg, 0xF1000000u | kb);
            DWS_ADD(w_a);
          }
          tc_fence_after();
          const int nq = min(GEMM_BK, t.Kc - kb * GEMM_BK) >> 4;
          const uint32_t alo = lo0 + smem0 + s * stage16, blo = alo + (GEMM_A_STAGE_BYTES >> 4);
          for (int q = 0; q < nq; ++q) umma_issue(tacc, alo + q * 16, hi, blo + q * 16, hi, idesc, (kb | q) ? 1u : 0u);
          umma_commit_1t(&op_empty[s]);
        }
        if (t.nkb > 0)
          umma_commit_1t(&acc_full[a]);
        else
          mbar_arrive(&acc_full[a]);
        ++j;
      }
    }
    __syncwarp();
  } else {
    // ===================== epilogue: Adam on the staged state =====================
    const int w = warp - 4, q = w & 3, g = w >> 2;
    const int kl = q * 32 + lane;          // tile-local input feature = TMEM lane
    const int et = threadIdx.x - 128;      // 0 .. 511
    uint32_t it = 0, j = 0;
    for (int tile = p.tile_begin + blockIdx.x; tile < p.tile_end; tile += gridDim.x) {
      const DwaTile t = dwa_tile(p, L, tile);
      if (!t.active) continue;
      const DwaLayer& y = L[t.layer];
      const AdamHyper h = adam_of(p.adam, p.adam_ms, t.model);
      const uint32_t a = j & 1, aph = (j >> 1) & 1;
      const int kk = t.m0 + kl;  // D row
      const bool is_w = kk < y.kin, is_b = kk == y.kin, is_c = kk > y.kin && kk < y.kaug;
      const int scol = is_w ? kl : kl - 1;  // shared-memory column of this thread's parameter (class columns: k - 1)
      const bool bias_tile = t.m0 <= y.kin && y.kin < t.m0 + GEMM_BM;
      const int* tab = p.tabs + y.tab_off;
      float* P = p.adam_p + t.model * p.state_ms;
      float* M1 = p.adam_m + t.model * p.state_ms;
      float* V2 = p.adam_v + t.model * p.state_ms;
      if (bias_tile) {
        if (et < t.BN) {
          const int srow = t.n0 + et;
          const int bo = srow < y.rcap ? tab[y.rcap + srow] : -1;
          bidx[et] = bo;
          bst[et] = bo >= 0 ? ld_global_f32(P + bo) : 0.f;
          bst[256 + et] = bo >= 0 ? ld_global_f32(M1 + bo) : 0.f;
          bst[512 + et] = bo >= 0 ? ld_global_f32(V2 + bo) : 0.f;
        }
        epi_bar_sync();
      }
      const bool have_acc = t.nkb > 0;
      if (lane == 0) {
        DWS_T0();
        mbar_wait_sleepy(&acc_full[a], aph, p.dbg, 0xA1000000u | tile);
        DWS_ADD(w_a);
      }
      __syncwarp();
      tc_fence_after();
      const uint32_t taddr = tmem_base + a * 256 + ((uint32_t)(q * 32) << 16) + g * DWA_RPW;
      // All epilogue warps work on the same stage (DWA_RPW weight rows each): a stage is occupied for the shortest
      // possible time, which is what the 4-slot ring needs.  Measured alternatives (profiles/r02_experiments.md): column
      // group g owning slot g and all 16 rows of its stages: 443 -> 503 us; writing p, m, v straight from registers
      // instead of tensor stores: 443 -> 475 us (that variant is gone).  The kernel is instruction-issue bound
      // (ncu: 56 % issue-active with 5 warps per scheduler), so the per-stage bookkeeping is kept out of this loop:
      // (tensor, row) of a stage's first weight row is tracked incrementally — stages advance by 16 shadow rows and
      // the stacking blocks are multiples of 16.
      int blk = t.n0 / y.ilv_stride, rem = t.n0 - blk * y.ilv_stride;
      const int my_off = (g * DWA_RPW) * 128 + scol;  // this thread's first element inside a stage array
      const bool wc = is_w || is_c;
      const int ss_off = ((kl >> 3) * DWA_R + g * DWA_RPW) * 8 + (kl & 7);
      const int nsub = t.BN / DWA_R;
      for (int sub = 0; sub < nsub; ++sub, ++it, rem += DWA_R) {
        if (rem >= y.ilv_stride) rem -= y.ilv_stride, ++blk;
        const int which = rem >= y.ilv_block ? 1 : 0;
        const int n = blk * y.ilv_block + rem - which * y.ilv_block;
        const bool has = which < y.ntens && n < y.rows_each;
        const int s = it % DWA_NST;
        uint32_t accr[DWA_RPW];
        if (have_acc) tmem_ldN_issue<DWA_RPW>(taddr + sub * DWA_R, accr);  // in flight while this warp waits for the stage
        if (lane == 0) {
          DWS_T0();
          mbar_wait_sleepy(&st_full[s], (it / DWA_NST) & 1, p.dbg, 0xA2000000u | sub);
          DWS_ADD(w_b);
        }
        __syncwarp();
        uint8_t* st = st_ring + (size_t)s * DWA_ST_STAGE;
        float* sp = reinterpret_cast<float*>(st) + my_off;
        float* sm = reinterpret_cast<float*>(st + DWA_ARR) + my_off;
        float* sv = reinterpret_cast<float*>(st + 2 * DWA_ARR) + my_off;
        bf16* ss = reinterpret_cast<bf16*>(st + 3 * DWA_ARR) + ss_off;
        float pv[DWA_RPW], mv[DWA_RPW], vv[DWA_RPW], acc[DWA_RPW];
        const bool upd = has && wc;
        if (upd) {
#pragma unroll
          for (int i = 0; i < DWA_RPW; ++i) pv[i] = sp[i * 128], mv[i] = sm[i * 128], vv[i] = sv[i * 128];
        }
        tmem_ldN_wait<DWA_RPW>(have_acc, accr, acc);  // warp-collective: outside the lane-dependent branches
        if (upd) {
#pragma unroll
          for (int i = 0; i < DWA_RPW; ++i) adam_update(acc[i], pv[i], mv[i], vv[i], h);
#pragma unroll
          for (int i = 0; i < DWA_RPW; ++i) sp[i * 128] = pv[i], sm[i * 128] = mv[i], sv[i * 128] = vv[i];
          if (!is_w) {  // class columns: the forward reads them as fp32 per-class bias rows
            float* d = p.drv + t.model * p.drv_ms + y.drv_clsb_off + (long long)(kk - y.kin - 1) * y.drv_clsb_ld + t.n0 + sub * DWA_R +
                       g * DWA_RPW;
#pragma unroll
            for (int i = 0; i < DWA_RPW; ++i)
              if (n + g * DWA_RPW + i < y.rows_each) d[i] = pv[i];
          }
        } else if (has && is_b) {
#pragma unroll
          for (int i = 0; i < DWA_RPW; ++i) {
            const int c = sub * DWA_R + g * DWA_RPW + i;  // tile-local weight row
            float pb = bst[c], mb = bst[256 + c], vb = bst[512 + c];
            adam_update(acc[i], pb, mb, vb, h);
            bst[c] = pb, bst[256 + c] = mb, bst[512 + c] = vb;
          }
        }
        // shadow stage [16 chunks][R rows][8]: columns >= kin (ones / class columns, padding) stay zero.  The four
        // 8-lane groups of a warp write four chunks 256 bytes apart, i.e. a 4-way bank conflict per store; that costs
        // shared-memory cycles the kernel has to spare, whereas the conflict-free rotated order cost DWA_RPW^2 selects
        // per stage on the resource it is short of (issue slots)
        const bool shw = upd && is_w;
#pragma unroll
        for (int i = 0; i < DWA_RPW; ++i) ss[i * 8] = __float2bfloat16_rn(shw ? pv[i] : 0.f);
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&st_done[s]);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[a]);
      if (bias_tile) {
        epi_bar_sync();
        if (et < t.BN) {
          const int bo = bidx[et];
          if (bo >= 0) {
            const float pv = bst[et];
            P[bo] = pv;
            M1[bo] = bst[256 + et];
            V2[bo] = bst[512 + et];
            p.drv[t.model * p.drv_ms + y.drv_bias_off + t.n0 + et] = pv + __int_as_float(tab[2 * y.rcap + t.n0 + et]);
          }
        }
        epi_bar_sync();  // the next bias tile may overwrite the staging arrays
      }
      ++j;
    }
  }
  if (STATS && p.stats && lane == 0) {
    if (warp == 0) atomicAdd(p.stats + DWS_PROD_EMPTY, (unsigned long long)w_a);
    if (warp == 1) atomicAdd(p.stats + DWS_LOADER_EMPTY, (unsigned long long)w_a);
    if (warp == 2) atomicAdd(p.stats + DWS_STORER_DONE, (unsigned long long)w_a), atomicAdd(p.stats + DWS_STORER_READ, (unsigned long long)w_b);
    if (warp == 4) atomicAdd(p.stats + DWS_EPI_ACC, (unsigned long long)w_a), atomicAdd(p.stats + DWS_EPI_STATE, (unsigned long long)w_b);
  }
  tc_fence_before();
  __syncthreads();
  if (STATS && p.stats && threadIdx.x == 0) atomicAdd(p.stats + DWS_CTA_TOTAL, (unsigned long long)(clock64() - cta_t0));
  if (warp == 3) tmem_dealloc(tmem_base, 512);
}

// fp32 tensor map of one weight tensor's optimizer-state array: {ld floats, rows, models}, box {128, DWA_R, 1}
inline cudaError_t dwa_state_map(CUtensorMap* out, float* base, int ld, int rows, long long model_stride, int n_models) {
  void* fp = nullptr;
  cudaDriverEntryPointQueryResult qr;
  cudaError_t err = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fp, cudaEnableDefault, &qr);
  if (err != cudaSuccess) return err;
  if (!fp || qr != cudaDriverEntryPointSuccess) return cudaErrorNotSupported;
  if ((ld & 3) || (model_stride & 3) || (reinterpret_cast<uintptr_t>(base) & 15)) return cudaErrorInvalidValue;
  const cuuint64_t dims[3] = {(cuuint64_t)ld, (cuuint64_t)rows, (cuuint64_t)(n_models < 1 ? 1 : n_models)};
  const cuuint64_t strides[2] = {(cuuint64_t)ld * 4, (cuuint64_t)(n_models > 1 ? model_stride : (long long)ld * rows) * 4};
  const cuuint32_t box[3] = {128, (cuuint32_t)DWA_R, 1};
  const cuuint32_t es[3] = {1, 1, 1};
  CUresult r = ((TmapEncodeFn)fp)(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                  CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? cudaSuccess : cudaErrorInvalidValue;
}

inline cudaError_t dwadam_launch(const DwaParams& p, cudaStream_t st, int max_ctas = 0) {
  static bool attr_set[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && !attr_set[dev]) {
    cudaError_t err = cudaFuncSetAttribute(dwadam_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, DWA_SMEM);
    if (err == cudaSuccess) err = cudaFuncSetAttribute(dwadam_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, DWA_SMEM);
    if (err != cudaSuccess) return err;
    attr_set[dev] = true;
  }
  int grid = std::min(p.tile_end - p.tile_begin, gemm_num_sms());
  if (max_ctas > 0) grid = std::min(grid, max_ctas);
  if (grid < 1) return cudaSuccess;
  if (p.stats) return launch_k(dwadam_kernel<true>, dim3(grid), dim3(DWA_THREADS), (size_t)DWA_SMEM, st, p);
  return launch_k(dwadam_kernel<false>, dim3(grid), dim3(DWA_THREADS), (size_t)DWA_SMEM, st, p);
}

}  // namespace drvae
