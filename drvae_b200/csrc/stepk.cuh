// Persistent step kernel: the whole forward + ELBO + input-gradient chain of one training / loss step as ONE
// cooperative launch (reference: the ~30-stage dependent chain of DrVAE._compute_losses / _fprop, src/DrVAE.py:333-543,
// and its autograd backward, src/DGMMixin.py:116-123; same for src/PVAE.py:265-409 and src/VFAE.py:234-401).
//
// Why.  As separate launches the chain is ~30 dependent kernels, each 6-25 us of launch latency, prologue (TMEM
// allocation, barrier init, descriptor fetch) and pipeline ramp for <= 10 us of work: 0.55 ms of a 1.0 ms ensemble step
// and nearly all of a single-model step (profiles/r02_experiments.md).  Here one CTA per SM stays resident for the
// whole chain: TMEM, the operand ring and its mbarriers are set up once, and the dependent stages are separated by a
// grid-wide barrier (~2 us) instead of a kernel boundary.
//
// How.  plan.cu still walks the step exactly as before (run_step), but its launches are RECORDED instead of issued:
// every GEMM (problem + epilogue parameters + tensor maps) and every row operation becomes an op with a level =
// 1 + the level of what it waits for, derived from the very stream / event dependencies the multi-launch schedule
// uses (main chain and label-dependent side branch).  The ops of one level — e.g. the decoder-loss GEMM of the main
// chain together with a small GEMM of the side branch — are cut into items (GEMM tiles, blocks of 16 rows) that the
// CTAs take round-robin; a grid barrier ends the level.  The device code of an item is the code of the stand-alone
// kernels: the warp-specialised tcgen05 mainloop and fused epilogues of gemm.cuh, the row functions of rowops.cuh.
//
// Roles per CTA (20 warps): warp 0 TMA producer, warp 3 MMA issuer, warps 4-19 epilogue of GEMM items and the workers
// of row items (one warp per row); warps 1-2 idle.  Operand ring: 4 stages x 48 KB; two 256-column TMEM accumulators.
#pragma once

#include <string>
#include <vector>

#include "rowops.cuh"

namespace drvae {

constexpr int STEPK_MAX_GEMM = 30;
constexpr int STEPK_MAX_OPS = 64;
constexpr int STEPK_MAX_LEVELS = 48;
constexpr int STEPK_STAGES = 4;
constexpr int STEPK_STAGE_BYTES = GEMM_A_STAGE_BYTES + 256 * GEMM_BK * 2;  // 48 KB: A tile + the widest B tile
// (dynamic shared memory: the ring + 1 KB alignment slack + the op tables, see step_kernel_launch)
constexpr int STEPK_THREADS = GEMM_THREADS;
constexpr int STEPK_ROWS = GEMM_EPI_WARPS;  // rows per row item: one per epilogue warp
constexpr int STEPK_ACC_COLS = 256;

enum { SOP_GEMM = 0, SOP_ROW = 1 };
enum {
  SROW_SAMPLE_Q1 = 0,
  SROW_T_POST,
  SROW_Z3_POST,
  SROW_PZ1_POST,
  SROW_Z3_BACK,
  SROW_CLF_BACK,
  SROW_T_BACK,
  SROW_Q_BACK,
  SROW_CLF_GRAD_PARTIAL,
  SROW_CLF_GRAD_REDUCE,
  SROW_LOSS_PARTIAL,
  SROW_LOSS_FINAL,
  SROW_CLF_FWD,
  SROW_CLF_DU,
  SROW_CLF_U,
  SROW_CLF_BACK_H,
  SROW_CLF_GRAD_PARTIAL_H
};

struct StepOp {
  int kind;        // SOP_*
  int sub;         // GEMM: epilogue (EPI_*); row op: SROW_*
  int idx;         // GEMM: index into StepParams::gemm / maps
  int item_begin;  // first item of this op inside its level
  int items;
  int per_model;   // row op: items per ensemble member
  int arg;         // row op: kernel-specific (loss slices)
};

struct StepGemm {
  GemmProblem p;
  EpiParams e;
};

// The op tables: kernel parameters on the way in, copied to shared memory by the first instructions of every CTA.
// (Read in place they cost a constant-cache miss per 64 bytes and level: the 30 KB parameter block is far larger than
// that cache, and every role touches a dozen lines of it per tile.)
struct StepTables {
  DevView v;
  int n_levels, n_ops;
  int level_op[STEPK_MAX_LEVELS + 1];
  int level_items[STEPK_MAX_LEVELS];
  StepOp ops[STEPK_MAX_OPS];
  StepGemm gemm[STEPK_MAX_GEMM];
};
static_assert(sizeof(StepTables) % 4 == 0, "copied word by word");

struct StepParams {
  StepTables t;
  alignas(64) CUtensorMap maps[3 * STEPK_MAX_GEMM];
  unsigned int* bar;  // {arrival count, generation}: self-resetting grid barrier
  DebugWord* dbg;
  unsigned long long* trace;  // kernel trace: one slot per level from trace_id0
  int trace_id0;
};
static_assert(sizeof(StepParams) <= 32000, "StepParams must fit the kernel parameter space");

// Grid barrier between two levels.  Writers (generic proxy stores of the epilogues / row functions) make their data
// visible to the TMA unit (async proxy) and to the other SMs before arriving; the wait is an acquire at gpu scope, so
// plain loads after it see the other CTAs' data (the cooperative-groups grid.sync() recipe).
__device__ __forceinline__ unsigned int ld_acquire_u32(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void step_grid_barrier(unsigned int* bar, DebugWord* dbg, int level, unsigned long long* trace_end) {
  asm volatile("fence.proxy.async;" ::: "memory");
  __syncthreads();
  if (threadIdx.x == 0) {
    if (trace_end) atomicMax(trace_end, global_ns());  // this CTA has finished the level
    __threadfence();
    const unsigned int gen = ld_acquire_u32(bar + 1);
    if (atomicAdd(bar, 1u) == gridDim.x - 1) {
      atomicExch(bar, 0u);
      __threadfence();
      atomicAdd(bar + 1, 1u);
    } else {
      const long long t0 = clock64();
      while (ld_acquire_u32(bar + 1) == gen) {
        __nanosleep(32);
        if (clock64() - t0 > 4000000000LL) {
          if (dbg) {
            dbg->code = 0xC0000000u | (unsigned)level;
            dbg->info[0] = blockIdx.x;
            __threadfence_system();
          }
          __trap();
        }
      }
    }
    __threadfence();
  }
  __syncthreads();
}

__device__ __forceinline__ const StepOp& step_find_op(const StepTables& P, int ob, int item) {
  int o = ob;
  while (item >= P.ops[o].item_begin + P.ops[o].items) ++o;
  return P.ops[o];
}

struct SyncNamed256 {  // warps 4-11 of the step kernel
  __device__ __forceinline__ void operator()() const { asm volatile("bar.sync 2, 256;" ::: "memory"); }
};

template <int EPI>
__device__ __forceinline__ void step_gemm_epilogue(const GemmProblem& p, const EpiParams& e, const TileInfo& t, uint32_t tmem_base,
                                                   uint32_t a, int q, int cg, int lane, bool have_acc) {
  RowCtx rc;
  rc.model = t.model;
  rc.row = t.m0 + q * 32 + lane;
  rc.cg = cg;
  rc.valid = rc.row < t.Mrows;
  const uint32_t taddr_row = tmem_base + a * STEPK_ACC_COLS + ((uint32_t)(q * 32) << 16);
  run_epilogue_row<EPI>(p, e, t, rc, taddr_row, have_acc, p.ksplit > 1);
}

__global__ void __launch_bounds__(STEPK_THREADS, 1) step_kernel(const __grid_constant__ StepParams PP) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[STEPK_STAGES];
  __shared__ __align__(8) uint64_t empty_bar[STEPK_STAGES];
  __shared__ __align__(8) uint64_t acc_full[GEMM_ACC_STAGES];
  __shared__ __align__(8) uint64_t acc_empty[GEMM_ACC_STAGES];
  __shared__ uint32_t tmem_base_s;
  __shared__ float loss_sm[256];

  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // op tables -> shared memory (after the ring)
  StepTables& T = *reinterpret_cast<StepTables*>(smem + STEPK_STAGES * STEPK_STAGE_BYTES);
  {
    const int* src = reinterpret_cast<const int*>(&PP.t);
    int* dst = reinterpret_cast<int*>(&T);
    for (int i = threadIdx.x; i < (int)(sizeof(StepTables) / 4); i += STEPK_THREADS) dst[i] = src[i];
  }

  if (threadIdx.x == 0) {
    for (int s = 0; s < STEPK_STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < GEMM_ACC_STAGES; ++a) {
      mbar_init(&acc_full[a], 1);
      mbar_init(&acc_empty[a], GEMM_EPI_WARPS);
    }
    mbar_fence_init();
  }
  if (warp == GEMM_MMA_WARP) {
    tmem_alloc(&tmem_base_s, GEMM_ACC_STAGES * STEPK_ACC_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;

  uint32_t ring_it = 0;  // k-blocks through the operand ring so far (producer and MMA warps count alike)
  uint32_t acc_j = 0;    // GEMM tiles of this CTA so far (MMA and epilogue warps count alike)

  for (int lv = 0; lv < T.n_levels; ++lv) {
    const int ob = T.level_op[lv], nitems = T.level_items[lv];
    if (PP.trace && threadIdx.x == 0) atomicMin(PP.trace + 2 * (long long)(PP.trace_id0 + lv), global_ns());

    if (warp == 1 && lv + 1 < T.n_levels) {
      // idle warp: descriptors of the next level's GEMMs into the TMA unit's cache while this level runs
      for (int o = T.level_op[lv + 1] + lane; o < T.level_op[lv + 2]; o += 32) {
        if (T.ops[o].kind == SOP_GEMM) {
          tma_prefetch_map(&PP.maps[3 * T.ops[o].idx]);
          tma_prefetch_map(&PP.maps[3 * T.ops[o].idx + 1]);
          tma_prefetch_map(&PP.maps[3 * T.ops[o].idx + 2]);
        }
      }
    }
    if (warp == 0) {
      // ===================== producer: TMA tensor loads of operand tiles =====================
      for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
        const StepOp& op = step_find_op(T, ob, item);
        if (op.kind != SOP_GEMM) continue;
        const GemmProblem& p = T.gemm[op.idx].p;
        const CUtensorMap* tm = &PP.maps[3 * op.idx];
        const TileInfo t = gemm_tile_info(p, item - op.item_begin);
        if (!t.active) continue;
        const bool a_mn = (p.mode == GEMM_DW), b_mn = (p.mode != GEMM_NT);
        const uint32_t stage_tx = GEMM_A_STAGE_BYTES + p.BN * GEMM_BK * 2;
        const bool b_split = !b_mn && p.BN > 128;
        for (int kb = t.kb_begin; kb < t.kb_end; ++kb, ++ring_it) {
          const int s = ring_it % STEPK_STAGES;
          const uint32_t ph = (ring_it / STEPK_STAGES) & 1;
          mbar_wait(&empty_bar[s], ph ^ 1, PP.dbg, 0xE0000000u | kb);
          uint8_t* As = smem + (size_t)s * STEPK_STAGE_BYTES;
          uint8_t* Bs = As + GEMM_A_STAGE_BYTES;
          if (elect_one()) {
            mbar_arrive_expect_tx(&full_bar[s], stage_tx);
            if (!a_mn)
              tma_load_3d(As, &tm[0], (p.A.row0 + t.m0) * 2, kb * 8, t.model, &full_bar[s]);
            else
              tma_load_3d(As, &tm[0], (p.A.row0 + kb * GEMM_BK) * 2, t.m0 >> 3, t.model, &full_bar[s]);
            if (!b_mn) {
              tma_load_3d(Bs, &tm[1], (p.B.row0 + t.n0) * 2, kb * 8, t.model, &full_bar[s]);
              if (b_split) tma_load_3d(Bs + 128 * GEMM_BK * 2, &tm[2], (p.B.row0 + t.n0 + 128) * 2, kb * 8, t.model, &full_bar[s]);
            } else {
              tma_load_3d(Bs, &tm[1], (p.B.row0 + kb * GEMM_BK) * 2, t.n0 >> 3, t.model, &full_bar[s]);
            }
          }
          __syncwarp();
        }
      }
    } else if (warp == GEMM_MMA_WARP) {
      // ===================== UMMA issuer (one elected lane; see gemm_tc_kernel) =====================
      if (elect_one()) {
        const uint32_t smem0 = smem_u32(smem) >> 4, stage16 = (uint32_t)STEPK_STAGE_BYTES >> 4;
        for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
          const StepOp& op = step_find_op(T, ob, item);
          if (op.kind != SOP_GEMM) continue;
          const GemmProblem& p = T.gemm[op.idx].p;
          const TileInfo t = gemm_tile_info(p, item - op.item_begin);
          if (!t.active) continue;
          const bool a_mn = (p.mode == GEMM_DW), b_mn = (p.mode != GEMM_NT);
          const int BN = p.BN;
          const bool b_split = !b_mn && BN > 128;
          const int bn0 = b_split ? 128 : BN, bn1 = BN - 128;
          const uint32_t idesc = umma_idesc_bf16(bn0, a_mn ? 1 : 0, b_mn ? 1 : 0);
          const uint32_t idesc1 = b_split ? umma_idesc_bf16(bn1, a_mn ? 1 : 0, 0) : 0u;
          uint32_t a_lbo, a_sbo, a_step, b_lbo, b_sbo, b_step;
          if (!a_mn) {
            a_lbo = GEMM_BM * 16, a_sbo = 128, a_step = 2 * GEMM_BM * 16;
          } else {
            a_lbo = 128, a_sbo = GEMM_BK * 16, a_step = 16 * 16;
          }
          if (!b_mn) {
            b_lbo = bn0 * 16, b_sbo = 128, b_step = 2 * bn0 * 16;
          } else {
            b_lbo = 128, b_sbo = GEMM_BK * 16, b_step = 16 * 16;
          }
          const uint32_t b1_lbo = bn1 * 16, b1_step = 2 * bn1 * 16;
          const uint64_t a_desc0 = umma_smem_desc(0, a_lbo, a_sbo), b_desc0 = umma_smem_desc(0, b_lbo, b_sbo);
          const uint64_t b1_desc0 = umma_smem_desc(0, b1_lbo, 128);
          const uint32_t a_hi = (uint32_t)(a_desc0 >> 32), b_hi = (uint32_t)(b_desc0 >> 32), b1_hi = (uint32_t)(b1_desc0 >> 32);
          const uint32_t a_lo0 = (uint32_t)a_desc0, b_lo0 = (uint32_t)b_desc0, b1_lo0 = (uint32_t)b1_desc0;
          const uint32_t da = a_step >> 4, db = b_step >> 4, db1 = b1_step >> 4;
          const uint32_t a = acc_j & 1, aph = (acc_j >> 1) & 1;
          mbar_wait(&acc_empty[a], aph ^ 1, PP.dbg, 0xB0000000u | item);
          tc_fence_after();
          const uint32_t tacc = tmem_base + a * STEPK_ACC_COLS;
          for (int kb = t.kb_begin; kb < t.kb_end; ++kb, ++ring_it) {
            const uint32_t s = ring_it % STEPK_STAGES, ph = (ring_it / STEPK_STAGES) & 1;
            mbar_wait(&full_bar[s], ph, PP.dbg, 0xF0000000u | kb);
            tc_fence_after();
            const int nq = min(GEMM_BK, t.Kc - kb * GEMM_BK) >> 4;
            const uint32_t sa = smem0 + s * stage16;
            const uint32_t alo = a_lo0 + sa, blo = b_lo0 + sa + (GEMM_A_STAGE_BYTES >> 4);
            const uint32_t b1lo = b1_lo0 + sa + ((GEMM_A_STAGE_BYTES + 128 * GEMM_BK * 2) >> 4);
            const uint32_t first = kb > t.kb_begin ? 1u : 0u;
            if (nq == 4 && !b_split) {
              umma_issue(tacc, alo, a_hi, blo, b_hi, idesc, first);
              umma_issue(tacc, alo + da, a_hi, blo + db, b_hi, idesc, 1u);
              umma_issue(tacc, alo + 2 * da, a_hi, blo + 2 * db, b_hi, idesc, 1u);
              umma_issue(tacc, alo + 3 * da, a_hi, blo + 3 * db, b_hi, idesc, 1u);
            } else {
              for (int qq = 0; qq < nq; ++qq) {
                const uint32_t accum = (first | (uint32_t)qq) ? 1u : 0u;
                umma_issue(tacc, alo + qq * da, a_hi, blo + qq * db, b_hi, idesc, accum);
                if (b_split) umma_issue(tacc + 128, alo + qq * da, a_hi, b1lo + qq * db1, b1_hi, idesc1, accum);
              }
            }
            umma_commit_1t(&empty_bar[s]);
          }
          if (t.kb_end > t.kb_begin)
            umma_commit_1t(&acc_full[a]);
          else
            mbar_arrive(&acc_full[a]);
          ++acc_j;
        }
      }
      __syncwarp();
    } else if (warp >= GEMM_EPI_WARP0) {
      // ===================== epilogue warps: GEMM epilogues and row items =====================
      const int w = warp - GEMM_EPI_WARP0;
      const int q = warp & 3, cg = w >> 2;
      for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
        const StepOp& op = step_find_op(T, ob, item);
        const int local = item - op.item_begin;
        if (op.kind == SOP_GEMM) {
          const GemmProblem& p = T.gemm[op.idx].p;
          const EpiParams& e = T.gemm[op.idx].e;
          const TileInfo t = gemm_tile_info(p, local);
          if (!t.active) continue;
          const uint32_t a = acc_j & 1, aph = (acc_j >> 1) & 1;
          const bool have_acc = t.kb_end > t.kb_begin;
          if (lane == 0) mbar_wait(&acc_full[a], aph, PP.dbg, 0xA0000000u | item);
          __syncwarp();
          tc_fence_after();
          switch (op.sub) {
            case EPI_STORE_F32: step_gemm_epilogue<EPI_STORE_F32>(p, e, t, tmem_base, a, q, cg, lane, have_acc); break;
            case EPI_ELU_C8: step_gemm_epilogue<EPI_ELU_C8>(p, e, t, tmem_base, a, q, cg, lane, have_acc); break;
            case EPI_DACT_C8: step_gemm_epilogue<EPI_DACT_C8>(p, e, t, tmem_base, a, q, cg, lane, have_acc); break;
            case EPI_DECLOSS: step_gemm_epilogue<EPI_DECLOSS>(p, e, t, tmem_base, a, q, cg, lane, have_acc); break;
            case EPI_GRAD: step_gemm_epilogue<EPI_GRAD>(p, e, t, tmem_base, a, q, cg, lane, have_acc); break;
            default: break;
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&acc_empty[a]);
          ++acc_j;
        } else {
          const int m = local / op.per_model;
          const int blk = local - (local / op.per_model) * op.per_model;
          const int r = blk * STEPK_ROWS + w;
          switch (op.sub) {
            case SROW_SAMPLE_Q1:
              if (T.v.Zc <= 128)
                sample_q1_row<4>(T.v, m, r, lane);
              else
                sample_q1_row<MAXJ>(T.v, m, r, lane);
              break;
            case SROW_T_POST:
              if (T.v.Zc <= 128)
                T_post_row<4>(T.v, m, r, lane);
              else
                T_post_row<MAXJ>(T.v, m, r, lane);
              break;
            case SROW_CLF_FWD: clf_fwd_row(T.v, m, r, lane); break;
            case SROW_Z3_POST: 
              if (T.v.Z3c <= 128)
                z3_post_row<4>(T.v, m, r, lane);
              else
                z3_post_row<MAXJ>(T.v, m, r, lane);
              break;
            case SROW_PZ1_POST: 
              if (T.v.Zc <= 128)
                pz1_post_row<4>(T.v, m, r, lane);
              else
                pz1_post_row<MAXJ>(T.v, m, r, lane);
              break;
            case SROW_Z3_BACK: 
              if (T.v.Z3c <= 128)
                z3_back_row<4>(T.v, m, r, lane);
              else
                z3_back_row<MAXJ>(T.v, m, r, lane);
              break;
            case SROW_CLF_BACK: clf_back_row(T.v, m, r, lane); break;
            case SROW_CLF_DU: clf_du_row(T.v, m, r, lane); break;
            case SROW_CLF_U: clf_u_row(T.v, m, r, lane); break;
            case SROW_CLF_BACK_H: clf_back_h_row(T.v, m, r, lane); break;
            case SROW_CLF_GRAD_PARTIAL_H: clf_grad_partial_h_block(T.v, m, blk, threadIdx.x - GEMM_EPI_WARP0 * 32, GEMM_EPI_WARPS * 32); break;
            case SROW_T_BACK: 
              if (T.v.Zc <= 128)
                T_back_row<4>(T.v, m, r, lane);
              else
                T_back_row<MAXJ>(T.v, m, r, lane);
              break;
            case SROW_Q_BACK: 
              if (T.v.Zc <= 128)
                q_back_row<4>(T.v, m, r, lane);
              else
                q_back_row<MAXJ>(T.v, m, r, lane);
              break;
            case SROW_CLF_GRAD_PARTIAL: clf_grad_partial_block(T.v, m, blk, threadIdx.x - GEMM_EPI_WARP0 * 32, GEMM_EPI_WARPS * 32); break;
            case SROW_CLF_GRAD_REDUCE: clf_grad_reduce_elem(T.v, m, r, lane); break;
            case SROW_LOSS_PARTIAL:
              if (w < 8) loss_partial_block(T.v, m, blk, op.arg, threadIdx.x - GEMM_EPI_WARP0 * 32, loss_sm, SyncNamed256());
              break;
            case SROW_LOSS_FINAL:
              if (w == 0 && lane == 0) loss_final_model(T.v, m);
              break;
            default: break;
          }
          __syncwarp();
        }
      }
    }
    unsigned long long* trace_end = PP.trace ? PP.trace + 2 * (long long)(PP.trace_id0 + lv) + 1 : nullptr;
    if (lv + 1 < T.n_levels) {
      step_grid_barrier(PP.bar, PP.dbg, lv, trace_end);
    } else if (trace_end) {
      __syncthreads();
      if (threadIdx.x == 0) atomicMax(trace_end, global_ns());
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == GEMM_MMA_WARP) tmem_dealloc(tmem_base, GEMM_ACC_STAGES * STEPK_ACC_COLS);
}

// ---------------------------------------------------------------------------------------------
// Host side: records the ops of one step and turns them into levels
// ---------------------------------------------------------------------------------------------
struct StepRecorder {
  struct Rec {
    StepOp op;
    int level;
    StepGemm g;
    std::string tag;
  };
  std::vector<Rec> recs;
  std::vector<cudaStream_t> streams;
  std::vector<int> cur;  // level of the last op per stream
  std::vector<std::pair<cudaEvent_t, int>> events;
  int n_gemm = 0;
  bool unsupported = false;

  int sid(cudaStream_t s) {
    for (size_t i = 0; i < streams.size(); ++i)
      if (streams[i] == s) return (int)i;
    streams.push_back(s);
    cur.push_back(0);
    return (int)streams.size() - 1;
  }
  void record_event(cudaEvent_t ev, cudaStream_t s) {
    const int l = cur[sid(s)];
    for (auto& e : events)
      if (e.first == ev) {
        e.second = l;
        return;
      }
    events.push_back({ev, l});
  }
  void wait_event(cudaStream_t s, cudaEvent_t ev) {
    const int i = sid(s);
    for (auto& e : events)
      if (e.first == ev) cur[i] = std::max(cur[i], e.second);
  }
  void after(cudaStream_t waiter, cudaStream_t producer) {
    const int w = sid(waiter), p = sid(producer);
    cur[w] = std::max(cur[w], cur[p]);
  }
  void add_gemm(int epi, const GemmProblem& p, const EpiParams& e, int n_models, cudaStream_t s, const std::string& tag) {
    if (epi != EPI_STORE_F32 && epi != EPI_ELU_C8 && epi != EPI_DACT_C8 && epi != EPI_DECLOSS && epi != EPI_GRAD) unsupported = true;
    if (p.BN > 256) unsupported = true;
    Rec r{};
    r.op.kind = SOP_GEMM;
    r.op.sub = epi;
    r.op.idx = n_gemm++;
    r.g.p = p;
    r.g.p.n_models = n_models;
    r.g.p.trace = nullptr;
    r.g.e = e;
    r.op.items = p.tiles_m * p.tiles_n * p.ksplit * n_models;
    const int i = sid(s);
    r.level = ++cur[i];
    r.tag = tag;
    recs.push_back(r);
  }
  void add_row(int kind, int per_model, int n_models, int arg, cudaStream_t s, const std::string& tag) {
    Rec r{};
    r.op.kind = SOP_ROW;
    r.op.sub = kind;
    r.op.per_model = per_model < 1 ? 1 : per_model;
    r.op.items = r.op.per_model * n_models;
    r.op.arg = arg;
    const int i = sid(s);
    r.level = ++cur[i];
    r.tag = tag;
    recs.push_back(r);
  }

  // -> parameter block; tags[l] names the ops of level l
  cudaError_t finalize(StepParams& P, std::vector<std::string>& tags, int& max_items) {
    if (unsupported || n_gemm > STEPK_MAX_GEMM || (int)recs.size() > STEPK_MAX_OPS || recs.empty()) return cudaErrorNotSupported;
    int nl = 0;
    for (auto& r : recs) nl = std::max(nl, r.level);
    if (nl > STEPK_MAX_LEVELS) return cudaErrorNotSupported;
    P.t.n_levels = nl;
    P.t.n_ops = (int)recs.size();
    tags.assign(nl, "");
    int o = 0;
    max_items = 1;
    for (int l = 1; l <= nl; ++l) {
      P.t.level_op[l - 1] = o;
      int items = 0;
      // small ops first: their items go to the first CTAs while the big GEMM of the level fills the rest
      std::vector<const Rec*> here;
      for (auto& r : recs)
        if (r.level == l) here.push_back(&r);
      std::stable_sort(here.begin(), here.end(), [](const Rec* a, const Rec* b) { return a->op.items < b->op.items; });
      for (const Rec* r : here) {
        StepOp op = r->op;
        op.item_begin = items;
        items += op.items;
        if (op.kind == SOP_GEMM) {
          P.t.gemm[op.idx] = r->g;
          cudaError_t err = gemm_make_maps(r->g.p, r->g.p.n_models, &P.maps[3 * op.idx], &P.maps[3 * op.idx + 1], &P.maps[3 * op.idx + 2]);
          if (err != cudaSuccess) return err;
        }
        P.t.ops[o++] = op;
        tags[l - 1] += (tags[l - 1].empty() ? "" : "+") + r->tag;
      }
      P.t.level_items[l - 1] = items;
      max_items = std::max(max_items, items);
    }
    P.t.level_op[nl] = o;
    return cudaSuccess;
  }
};

constexpr int STEPK_SMEM = STEPK_STAGES * STEPK_STAGE_BYTES + 1024 + (int)sizeof(StepTables);
static_assert(STEPK_SMEM + 4096 <= 227 * 1024, "ring + op tables + static shared memory must fit one SM");

inline cudaError_t step_kernel_launch(const StepParams& P, int max_items, cudaStream_t st) {
  static bool attr_set[64] = {};
  const int dev = gemm_current_device();
  if (!attr_set[dev]) {
    cudaError_t err = cudaFuncSetAttribute(step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, STEPK_SMEM);
    if (err != cudaSuccess) return err;
    attr_set[dev] = true;
  }
  const int grid = std::max(1, std::min(gemm_num_sms(), max_items));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(STEPK_THREADS);
  cfg.dynamicSmemBytes = STEPK_SMEM;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeCooperative;  // every CTA resident at once: the grid barrier needs it
  attr[0].val.cooperative = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, step_kernel, P);
}

}  // namespace drvae
