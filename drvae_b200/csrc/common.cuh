// Shared device helpers for the drvae_b200 kernels (sm_100a only).
//
// Everything here is plumbing for the hot path named in SURVEY.md §8: PTX wrappers for
// mbarrier / bulk-copy (TMA) / tcgen05 (TMEM + UMMA), the "chunk8" operand layout, and the
// watchdog that turns a would-be hang into a trapped, reported error.
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <utility>

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "drvae_b200 kernels are written for sm_100a (B200) only"
#endif

namespace drvae {

typedef __nv_bfloat16 bf16;

// ---------------------------------------------------------------------------------------------
// chunk8 layout.  Every GEMM operand (activations, pre-activation gradients, bf16 weight
// shadows) lives in HBM as  buf[feature/8][row][feature%8]  (bf16), i.e. one 16-byte "atom" per
// (row, 8-feature chunk), rows contiguous inside a chunk.  `rcap` is the row capacity (row
// stride between chunks).  A [rows x 8k] slab of this buffer is already the no-swizzle UMMA
// canonical layout, K-major when the contraction runs over features and MN-major when it runs
// over rows, so one storage format feeds forward, dX and dW GEMMs: a tile is one TMA box of a 3-D tensor map over
// {row x 16 B, feature chunk, model} (gemm.cuh, gemm_c8_map).
// ---------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ long long c8_index(int row, int feat, int rcap) {
  return ((long long)(feat >> 3) * rcap + row) * 8 + (feat & 7);
}

// Device error word: kernels write a code here before trapping so the host can say what hung.
struct DebugWord {
  unsigned int code;
  unsigned int info[7];
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}

// Kernel launch that returns the launch's error status.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

// ---------------------------------------------------------------------------------------------
// Kernel trace (drvae_trace_begin / _end): every kernel of the step stamps %globaltimer when its first CTA starts and
// when its last CTA leaves, into slot `id` of a device buffer.  The host turns the slots into a timeline of the step
// as it really ran (streams overlapping, launch gaps), which per-launch event brackets cannot show.  Off (null
// buffer) it costs one predictable branch per CTA.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
struct TraceScope {
  unsigned long long* slot;
  __device__ __forceinline__ TraceScope(unsigned long long* buf, int id) : slot(buf ? buf + 2 * (long long)id : nullptr) {
    if (slot && threadIdx.x == 0) atomicMin(slot, global_ns());
  }
  __device__ __forceinline__ ~TraceScope() {
    if (slot && threadIdx.x == 0) atomicMax(slot + 1, global_ns());
  }
};

// ---------------------------------------------------------------------------------------------
// mbarrier
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// try_wait with a suspend-time hint: the thread may sleep in hardware up to `ns` nanoseconds waiting for the phase,
// instead of returning to a software polling loop after the (short) default time
__device__ __forceinline__ bool mbar_try_wait_hint(uint64_t* bar, uint32_t parity, uint32_t ns) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(ns)
      : "memory");
  return ok != 0;
}
// Bounded wait for long-running producers/consumers of a persistent kernel: hardware-suspended polling (few issued
// instructions while waiting), trap with a code after ~2 s.
__device__ __forceinline__ void mbar_wait_sleepy(uint64_t* bar, uint32_t parity, DebugWord* dbg, uint32_t code) {
  if (mbar_try_wait(bar, parity)) return;
  for (int spins = 0; !mbar_try_wait_hint(bar, parity, 2000u); ++spins) {
    if (spins > 1000000) {  // >= 2 s of suspended waiting
      if (dbg) {
        dbg->code = code;
        dbg->info[0] = blockIdx.x;
        dbg->info[3] = threadIdx.x;
        dbg->info[4] = parity;
        __threadfence_system();
      }
      __trap();
    }
  }
}
// Bounded wait: a barrier that never completes (wrong tx byte count, lost commit) becomes a
// trapped kernel with a code in the debug word instead of a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, DebugWord* dbg, uint32_t code) {
  if (mbar_try_wait(bar, parity)) return;
  long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    __nanosleep(40);  // back off: pollers must not starve the producer / MMA warps of issue slots
    if (clock64() - t0 > 4000000000LL) {  // ~2 s at 2 GHz
      if (dbg) {
        dbg->code = code;
        dbg->info[0] = blockIdx.x;
        dbg->info[1] = blockIdx.y;
        dbg->info[2] = blockIdx.z;
        dbg->info[3] = threadIdx.x;
        dbg->info[4] = parity;
        __threadfence_system();
      }
      __trap();
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Tensor load global -> shared of one 3-D box (TMA unit, SASS UTMALDG), completion on an mbarrier.  `map` must
// live in parameter (__grid_constant__), constant or global memory.
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const void* map, int c0, int c1, int c2, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
          smem_u32(smem_dst)),
      "l"((unsigned long long)map), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar))
      : "memory");
}

// Fetch a tensor map (kernel parameter) into the TMA unit's descriptor cache ahead of its first use.
__device__ __forceinline__ void tma_prefetch_map(const void* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"((unsigned long long)map) : "memory");
}

// ---------------------------------------------------------------------------------------------
// tcgen05: TMEM allocation, UMMA issue, commit, TMEM loads
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// One lane of a CONVERGED warp (elect.sync picks the same lane every time for a full mask).  The single-thread
// instructions below (tcgen05.mma / commit, TMA loads) are issued from warp-uniform code under this predicate:
// with uniform control flow and operands ptxas keeps descriptors and addresses in uniform registers, whereas the
// same instructions under `if (lane == 0)` are wrapped in a per-lane ELECT / R2UR.BROADCAST loop (~50 SASS
// instructions per MMA on the one thread the whole tile waits for).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
// D[tmem] (+)= A[smem] * B[smem], kind::f16 (bf16 in, fp32 accumulate): called by the whole (converged) warp, issued
// by its elected lane.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  if (elect_one()) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}
// Single-thread forms for an issue loop that already runs on one elected lane: descriptors as 32-bit halves (only
// the low word, which holds the shared-memory address, changes between MMAs), no election per instruction.  The
// issuing thread is the critical path of a tile: tools/umma_rate_bench.cu measures 128 cycles per N=256 MMA (the
// hardware floor) for back-to-back issue and 133-275 cycles when every MMA carries its own election and
// descriptor arithmetic.
__device__ __forceinline__ void umma_issue(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                           uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}" ::"r"(tmem_d),
      "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_1t(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// Arrive on an mbarrier once all UMMAs previously issued by the elected lane have completed (whole warp calls).
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  if (elect_one()) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
  }
}
// 32 lanes x 16 consecutive fp32 columns: thread t of the warp reads TMEM lane (lane_base + t).
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  __syncwarp();  // .sync.aligned: make sure the warp is converged after predicated epilogue stores
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// Two 16-column loads in flight before one wait (decoder heads: mu and sigma halves of a tile).
__device__ __forceinline__ void tmem_ld16x2(uint32_t taddr0, uint32_t taddr1, float (&v0)[16], float (&v1)[16]) {
  uint32_t r[16], q[16];
  __syncwarp();
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr0)
      : "memory");
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(q[0]), "=r"(q[1]), "=r"(q[2]), "=r"(q[3]), "=r"(q[4]), "=r"(q[5]), "=r"(q[6]), "=r"(q[7]),
        "=r"(q[8]), "=r"(q[9]), "=r"(q[10]), "=r"(q[11]), "=r"(q[12]), "=r"(q[13]), "=r"(q[14]), "=r"(q[15])
      : "r"(taddr1)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    v0[i] = __uint_as_float(r[i]);
    v1[i] = __uint_as_float(q[i]);
  }
}

// UMMA shared-memory matrix descriptor, no-swizzle ("interleave") canonical layout.
// Field meaning follows cute::UMMA::SmemDescriptor (start>>4 | LBO>>4 @16 | SBO>>4 @32 |
// version=1 @46 | layout_type=0 @61).  For a K-major operand SBO is the byte distance between
// 8-row groups and LBO between the two 8-element K halves of one K=16 step; for an MN-major
// operand SBO is the distance between 8-element MN chunks and LBO between 8-row K groups.
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFFu);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}
// UMMA instruction descriptor (cute::UMMA::InstrDescriptor): fp32 accumulate, bf16 A and B,
// majors selectable, M = 128, N = bn.
__device__ __forceinline__ uint32_t umma_idesc_bf16(int bn, int a_mn_major, int b_mn_major) {
  uint32_t d = 0;
  d |= 1u << 4;                       // c_format = F32
  d |= 1u << 7;                       // a_format = BF16
  d |= 1u << 10;                      // b_format = BF16
  d |= (uint32_t)(a_mn_major & 1) << 15;
  d |= (uint32_t)(b_mn_major & 1) << 16;
  d |= (uint32_t)(bn >> 3) << 17;     // n_dim
  d |= (uint32_t)(128 >> 4) << 24;    // m_dim
  return d;
}

// ---------------------------------------------------------------------------------------------
// small math helpers shared by epilogues and row kernels
// ---------------------------------------------------------------------------------------------
// ELU(alpha=1).  exp(x) - 1 with the fast exponential: the result is stored as bf16 (8 mantissa
// bits), so the cancellation error near 0 (~6e-8 absolute) is far below the storage rounding.
__device__ __forceinline__ float elu1(float x) { return x > 0.f ? x : __expf(x) - 1.f; }
// d ELU / d pre, recovered from the stored (bf16-rounded) activation h: 1 if h > 0 else h + 1.
__device__ __forceinline__ float elu1_grad_from_out(float h) { return h > 0.f ? 1.f : h + 1.f; }
// Softplus hidden layers (torch.nn.Softplus(): log1p(exp(x)), x for x > 20), stored as bf16.  The result has to keep
// bf16's RELATIVE precision for x << 0, where softplus(x) ~ exp(x) is tiny: exp(x) without flush-to-zero (exact down to
// the denormal range), then log1p(e) as e (1 - e (1/2 - e (1/3 - e/4))) for e < 1/16 (relative error < e^4 / 5 < 4e-6)
// and as lg2(1 + e) ln 2 above (1 + e rounds e to 2^-24 absolute, < 3e-7 relative there).  One ex2 and one lg2 per
// element.
__device__ __forceinline__ float softplus_act(float x) {
  const float LOG2E = 1.4426950408889634f, LN2 = 0.6931471805599453f;
  float e, l;
  asm("ex2.approx.f32 %0, %1;" : "=f"(e) : "f"(fminf(x, 20.f) * LOG2E));
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"(1.f + e));
  const float small = e * fmaf(e, fmaf(e, fmaf(e, -0.25f, 1.f / 3.f), -0.5f), 1.f);
  return x > 20.f ? x : (e < 0.0625f ? small : l * LN2);
}
// d softplus / d pre = sigmoid(x), recovered from the stored (bf16-rounded) activation h as -expm1(-h): h (1 - h (1/2 -
// h (1/6 - h/24))) for h < 1/16, where 1 - exp(-h) would cancel (h ~ exp(x) is tiny for x << 0 but carries bf16
// relative precision; series error < h^4 / 120), 1 - exp(-h) above, 1 for h > 20.
__device__ __forceinline__ float softplus_grad_from_out(float h) {
  const float small = h * fmaf(h, fmaf(h, fmaf(h, -1.f / 24.f, 1.f / 6.f), -0.5f), 1.f);
  return h > 20.f ? 1.f : (h < 0.0625f ? small : 1.f - __expf(-h));
}
// torch.nn.Softplus(beta=1, threshold=20)
__device__ __forceinline__ float softplus20(float x) { return x > 20.f ? x : log1pf(expf(x)); }
__device__ __forceinline__ float sigmoid_sp(float x) { return x > 20.f ? 1.f : 1.f / (1.f + expf(-x)); }

// torch.optim.Adam with coupled weight decay (SURVEY.md Appendix A.6; reference DGMMixin.py:31-40):
//   g <- g + wd p ; m <- b1 m + (1-b1) g ; v <- b2 v + (1-b2) g^2 ;
//   p <- p - (lr / (1-b1^t)) * m / (sqrt(v) / sqrt(1-b2^t) + eps)
// One definition for the stand-alone optimizer kernel and the grouped dW+Adam kernel, so both
// apply bit-identical updates.  sqrt / divide use the hardware approximations (<= 2 ulp): the
// update is ~lr in magnitude, so the absolute effect is ~1e-10 per step.
struct AdamHyper {
  float lr_bc1, beta1, beta2, eps, wd, inv_sqrt_bc2;
};
// Adam scalars of global model `model`: `ms` bytes between models (0: one copy shared by the ensemble).
__device__ __forceinline__ AdamHyper adam_of(const AdamHyper* h, int ms, int model) {
  return *reinterpret_cast<const AdamHyper*>(reinterpret_cast<const char*>(h) + (long long)model * ms);
}
__device__ __forceinline__ void adam_update(float g, float& p, float& m, float& v, const AdamHyper& h) {
  const float gr = g + h.wd * p;
  m = h.beta1 * m + (1.f - h.beta1) * gr;
  v = h.beta2 * v + (1.f - h.beta2) * gr * gr;
  float s;
  asm("sqrt.approx.f32 %0, %1;" : "=f"(s) : "f"(v));
  // m / d as m * rcp.approx(d): d = sqrt(v) / sqrt(bc2) + eps lies far inside the normal range, so the range scaling of
  // __fdividef (4 more instructions per parameter in an issue-bound kernel) buys nothing
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(s * h.inv_sqrt_bc2 + h.eps));
  p = p - h.lr_bc1 * (m * r);
}

__device__ __forceinline__ void philox4x32_10(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
    const uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
    c[0] = n0;
    c[1] = n1;
    c[2] = n2;
    c[3] = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
}

// Four standard normals keyed by (seed, step, model, draw kind `seg`, MC sample l, GLOBAL row, quad q of the
// row): Philox4x32-10 + Box-Muller with the hardware approximations (noise: ~1e-6 absolute error is
// irrelevant); the clamp keeps -2 log(u) non-negative when u rounds to 1.
__device__ __forceinline__ void philox_normal4(unsigned long long seed, unsigned int step, int model, int seg, int l,
                                               unsigned long long grow, int q, float (&z)[4]) {
  uint32_t c[4] = {(uint32_t)q | ((uint32_t)(grow >> 32) << 24), (uint32_t)grow, step,
                   (uint32_t)model | ((uint32_t)seg << 20) | ((uint32_t)l << 24)};
  philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
  const float k = 2.3283064365386963e-10f;  // 2^-32
  const float u0 = (c[0] + 1.0f) * k, u1 = c[1] * k, u2 = (c[2] + 1.0f) * k, u3 = c[3] * k;
  float r0, r1;
  asm("sqrt.approx.f32 %0, %1;" : "=f"(r0) : "f"(fmaxf(-2.f * __logf(fminf(u0, 1.f)), 0.f)));
  asm("sqrt.approx.f32 %0, %1;" : "=f"(r1) : "f"(fmaxf(-2.f * __logf(fminf(u2, 1.f)), 0.f)));
  float s0, c0, s1, c1;
  __sincosf(6.283185307179586f * u1, &s0, &c0);
  __sincosf(6.283185307179586f * u3, &s1, &c1);
  z[0] = r0 * c0, z[1] = r0 * s0, z[2] = r1 * c1, z[3] = r1 * s1;
}

// Packed fp32 pairs (Blackwell FADD2 / FMUL2 / FFMA2: one issue slot for two IEEE-rounded fp32 operations).  For the
// epilogues that ncu shows bound by instruction issue rather than by a pipe.
__device__ __forceinline__ float2 add2(float2 a, float2 b) {
  unsigned long long ra, rb, rd;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
  float2 d;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(rd));
  return d;
}
__device__ __forceinline__ float2 mul2(float2 a, float2 b) {
  unsigned long long ra, rb, rd;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
  float2 d;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(rd));
  return d;
}
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) {
  unsigned long long ra, rb, rc, rd;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rc) : "f"(c.x), "f"(c.y));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
  float2 d;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(rd));
  return d;
}
__device__ __forceinline__ float2 splat2(float x) { return make_float2(x, x); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&p);
}
__device__ __forceinline__ void unpack_bf16x8(const uint4& q, float (&f)[8]) {
  const __nv_bfloat162* p = reinterpret_cast<const __nv_bfloat162*>(&q);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 t = __bfloat1622float2(p[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ uint4 pack_bf16x8(const float* f) {
  uint4 q;
  q.x = pack_bf16x2(f[0], f[1]);
  q.y = pack_bf16x2(f[2], f[3]);
  q.z = pack_bf16x2(f[4], f[5]);
  q.w = pack_bf16x2(f[6], f[7]);
  return q;
}

}  // namespace drvae
