// Grouped (one problem per ensemble member) GEMM on tcgen05 tensor cores with fused epilogues.
//
// One kernel template serves every linear layer of the DrVAE / PVAE / VFAE step
// (reference: src/blocks.py:95-164 MLP, :243-301 DiagGaussianModule, :304-361
// DiagGaussianModuleLinear, :364-416 DiagGaussianSigmaModule) in three contraction modes over
// the same chunk8 operand storage (see common.cuh):
//   GEMM_NT  forward        D[rows, out]  = X[rows, in]   . W[out, in]^T     (A, B K-major)
//   GEMM_DX  input grad     D[rows, in]   = dY[rows, out] . W[out, in]       (A K-major, B MN-major)
//   GEMM_DW  weight grad    D[in, out]    = X[rows, in]^T . dY[rows, out]    (A, B MN-major)
// The weight gradient is produced TRANSPOSED (D row = input feature, D column = output feature)
// so that the 32 lanes of an epilogue warp (32 consecutive D rows) touch 32 consecutive elements
// of a row of the reference's [out, in] weight tensor: gradient stores are 128-byte coalesced.  Every GEMM
// input carries a ones column (and the one-hot class columns of [z, onehot(y)] inputs) after its
// last real feature, so the bias and class-column gradients are rows of the same D tile.
// Operand tiles are moved global->shared by TMA tensor loads (one box per operand tile and
// k-block: a chunk8 buffer is described as a 3-D tensor {row x 16 B, feature chunk, model} of
// 8-byte elements, so a box lands in shared memory as the no-swizzle UMMA canonical layout),
// multiplied with tcgen05.mma (bf16 in, fp32 accumulate in TMEM) by one elected thread, and the
// accumulator tile is read back with tcgen05.ld by the epilogue warps that apply the layer's
// epilogue (bias/ELU, ELU', Gaussian log-density + its gradient, weight gradient, ...).  The weight gradients and
// Adam of a fused train step are not computed here but in the grouped launch of dwadam.cuh.
//
// A slow SIMT kernel with the *same* operand format and the *same* epilogue code is kept as a
// validation reference for the tensor-core mainloop (tests only; never selected implicitly).
#pragma once

#include <cuda.h>  // CUtensorMap (types only: the encoder is resolved through cudaGetDriverEntryPoint)

#include <map>
#include <mutex>
#include <tuple>

#include "common.cuh"

namespace drvae {

enum { GEMM_NT = 0, GEMM_DX = 1, GEMM_DW = 2 };

enum {
  EPI_STORE_F32 = 0,  // (+bias) -> fp32 row-major
  EPI_ELU_C8 = 1,     // +bias (+class bias) -> ELU -> bf16 chunk8
  EPI_DACT_C8 = 2,    // * ELU'(stored activation) -> bf16 chunk8
  EPI_GRAD = 3,       // weight (+bias, +class column) gradient -> flat fp32 grad buffer, reference tensor layout
  EPI_DECLOSS = 4,    // decoder heads: Gaussian log-density partials + d loss / d pre-activation
  EPI_DECOUT = 5      // decoder heads at inference: mu and sigma as fp32 row-major
};

constexpr int GEMM_BM = 128;
constexpr int GEMM_BK = 64;
constexpr int GEMM_MAX_STAGES = 8;
constexpr int GEMM_A_STAGE_BYTES = GEMM_BM * GEMM_BK * 2;  // 16 KB
constexpr int GEMM_EPI_WARPS = 16;                     // epilogue warps of the persistent kernel
constexpr int EPI_GROUPS = GEMM_EPI_WARPS / 4;         // column groups: a warp reads TMEM lanes 32*(warp%4).., columns of its group
constexpr int GEMM_PROD_WARPS = 3;                     // warps before the MMA warp: warp 0 is the TMA producer, warps 1-2 are idle
                                                       // (they issued bulk copies before the operands moved to tensor loads; the
                                                       // count keeps epilogue warp w on TMEM lane quarter w % 4)
constexpr int GEMM_MMA_WARP = GEMM_PROD_WARPS;         // warp 3: MMA issuer; warps 4.. epilogue
constexpr int GEMM_EPI_WARP0 = GEMM_PROD_WARPS + 1;
constexpr int GEMM_THREADS = (GEMM_PROD_WARPS + 1 + GEMM_EPI_WARPS) * 32;
constexpr int GEMM_SIMT_THREADS = 128 * EPI_GROUPS;    // validation kernel: thread = (row, column group)
constexpr int GEMM_ACC_STAGES = 2;                     // accumulator tiles in TMEM (epilogue of tile i overlaps mainloop of i+1)
constexpr int GEMM_SMEM_BUDGET = 208 * 1024;           // operand ring per CTA (one CTA per SM)

// Optional instrumentation (-DGEMM_PROFILE_WAITS, tools/wait_profile.py): cycles the producer / MMA / epilogue roles
// spend blocked on each mbarrier, summed per (mode, epilogue) over CTAs and launches.  Compiled out by default.
#ifdef GEMM_PROFILE_WAITS
static __device__ unsigned long long g_wait_stats[3 * 8 * 8];
#define WS_T0() const long long ws_t0 = clock64()
#define WS_ADD(c) atomicAdd(&g_wait_stats[(p.mode * 8 + EPI) * 8 + (c)], (unsigned long long)(clock64() - ws_t0))
#define WS_INC(c, v) atomicAdd(&g_wait_stats[(p.mode * 8 + EPI) * 8 + (c)], (unsigned long long)(v))
#else
#define WS_T0()
#define WS_ADD(c)
#define WS_INC(c, v)
#endif
enum { WS_PROD_EMPTY = 0, WS_MMA_FULL, WS_MMA_ACC_EMPTY, WS_EPI_ACC_FULL, WS_EPI_BUSY, WS_CTA_TOTAL, WS_TILES, WS_KBLOCKS };

struct GemmOperand {
  const bf16* base;        // model 0
  long long model_stride;  // elements between ensemble members
  int rcap;                // row capacity of the chunk8 buffer
  int nchunks;             // feature chunks that exist in the buffer
  int row0;                // first row of the view
};

struct GemmProblem {
  GemmOperand A, B;
  int mode;
  int M, N, K;      // static upper bounds of D rows / D cols / contraction length
  const int* dyn;   // per-model dynamic extent: rows of D (NT, DX) or contraction rows (DW); may be null
  int dyn_stride;   // ints between models in `dyn`
  int BN;           // N tile (multiple of 16, <= 256)
  int tiles_n;
  int tiles_m;
  int nstages;
  int ksplit;       // >1: contraction split into ksplit tiles (EPI_GRAD accumulates atomically)
  int n_models;     // models of this launch
  int ens;          // ensemble members the operand buffers hold (extent of the tensor maps); 0: n_models
  int desc_variant; // debug knob for descriptor bring-up (0 = designed encoding)
  int max_ctas;     // > 0: cap on the persistent grid (the step reserves SMs for a concurrent launch)
  DebugWord* dbg;
  unsigned long long* trace;  // kernel trace (common.cuh TraceScope)
  int trace_id;
};

struct EpiParams {
  // fp32 row-major output (EPI_STORE_F32, EPI_DECOUT mu)
  float* out_f32;
  long long out_f32_ms;
  int out_ld;
  int out_row0;
  // second fp32 output (EPI_DECOUT sigma)
  float* out2_f32;
  // bf16 chunk8 output
  bf16* out_c8;
  long long out_c8_ms;
  int out_c8_rcap;
  int out_c8_row0;
  int n_valid;  // valid output columns (features); chunk8 outputs get a ones column at n_valid
  // bias: derived fp32 vector of length >= tiles_n*BN (constant offsets folded in, zero padded)
  const float* bias;
  long long bias_ms;
  // per-class bias rows (one-hot y folded out of the forward GEMM): clsb[cls*clsb_ld + col]
  const float* clsb;
  long long clsb_ms;
  int clsb_ld;
  const int* row_cls;  // class of each D row
  long long row_cls_ms;
  // stored activation for EPI_DACT_C8 (same geometry as the chunk8 output)
  const bf16* act;
  long long act_ms;
  int act_rcap;
  int act_row0;
  // EPI_GRAD: D row = input feature k (k == g_kin: ones column -> bias gradient,
  // k > g_kin: one-hot class columns), D col = shadow row s.  g_tab holds three int tables of
  // g_tab_n entries each, indexed by s: flat offset of W[n(s)][0] (or -1: padding row), flat
  // offset of b[n(s)], and the constant folded into the derived bias (float bits).
  float* grad;
  long long grad_ms;
  const int* g_tab;
  int g_tab_n;
  int g_kin;      // true input features
  int g_kaug;     // g_kin + 1 + class columns
  // EPI_DECLOSS / EPI_DECOUT
  const float4* tgt4;  // fp32 targets, chunk4 layout [Xc/4][tgt_rcap] float4
  long long tgt_ms;    // float4 elements between models
  int tgt_rcap;
  int X;             // feature count of the data space
  int Xc;            // feature capacity of tgt4 (multiple of 16)
  const int* counts; // per-model counts block (CNT_*)
  int counts_stride;
  const float* coefs;  // per-model coefficient block (COEF_*)
  int coefs_stride;
  int L;
  float* part;  // [tiles_n * EPI_GROUPS][Rdcap] row partial log-densities
  long long part_ms;
  int part_rcap;
  int write_dy;  // 0 in eval mode (loss only)
};

// Offsets inside the per-model counts / coefficient blocks (written by rowmap_kernel).
enum { CNT_N = 0, CNT_NP, CNT_NLAB, CNT_R0, CNT_LN, CNT_RD, CNT_F, CNT_FL, CNT_LNP, CNT_SIZE = 16 };
enum {
  COEF_RECL = 0,  // 1 / (L * Nglobal)
  COEF_PERT,      // beta_pert * pertloss_rate / (L * max(1, Np_global))
  COEF_KLZ2,      // beta_pert * kl_qz2pz2_rate / (L * Nglobal)
  COEF_KLD,       // 1 / (L * Nglobal)
  COEF_YL,        // beta_yr * yloss_rate / (L * max(1, Nlab_global))
  COEF_INV_N,       // 1 / Nglobal
  COEF_PERT_PLAIN,  // 1 / (L * max(1, Np_global))
  COEF_YL_PLAIN,    // 1 / (L * max(1, Nlab_global))
  COEF_SIZE = 16
};

struct RowCtx {
  int model;
  int row;     // D row (global within the problem)
  int cg;      // column group of the calling warp (0 .. EPI_GROUPS-1)
  bool valid;  // row < dynamic extent
  int cls;
  // DECLOSS
  int trow;    // target row, -1: none
  float coef;
  float lsum;
};

// ---------------------------------------------------------------------------------------------
// Epilogue pieces (shared by the tensor-core and the SIMT validation kernels).  Each call handles
// 16 consecutive D columns [col0, col0+16) of one D row held by the calling thread.
// ---------------------------------------------------------------------------------------------
template <int EPI>
__device__ __forceinline__ void epi_begin(const EpiParams& e, RowCtx& rc) {
  rc.cls = 0;
  rc.lsum = 0.f;
  rc.trow = -1;
  rc.coef = 0.f;
  if (EPI == EPI_ELU_C8) {
    if (e.row_cls && rc.valid) rc.cls = e.row_cls[rc.model * e.row_cls_ms + rc.row];
  }
  if (EPI == EPI_DECLOSS) {
    if (rc.valid) {
      const int* cnt = e.counts + (long long)rc.model * e.counts_stride;
      const float* cf = e.coefs + (long long)rc.model * e.coefs_stride;
      const int N = cnt[CNT_N], Np = cnt[CNT_NP];
      const int LN = e.L * N, LNp = e.L * Np;
      int t;
      float c;
      if (rc.row < LN) {
        t = rc.row % N;
        c = cf[COEF_RECL];
      } else if (rc.row < LN + LNp) {
        t = N + (rc.row - LN) % Np;
        c = cf[COEF_RECL];
      } else {
        t = N + (rc.row - LN - LNp) % Np;
        c = cf[COEF_PERT];
      }
      rc.trow = t;
      rc.coef = c;
    }
  }
}

__device__ __forceinline__ float ld_global_f32(const float* p) {
  float v;
  asm volatile("ld.global.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
  return v;
}

template <int EPI>
__device__ __forceinline__ void epi_chunk(const EpiParams& e, RowCtx& rc, int col0, float (&acc)[16], bool atomic) {
  if (EPI == EPI_STORE_F32) {
    if (!rc.valid) return;
    float* o = e.out_f32 + rc.model * e.out_f32_ms + (long long)(e.out_row0 + rc.row) * e.out_ld;
    const float* b = e.bias ? e.bias + rc.model * e.bias_ms : nullptr;
    if (((e.out_ld | e.n_valid) & 3) == 0) {
#pragma unroll
      for (int i = 0; i < 16; i += 4) {
        const int c = col0 + i;
        if (c < e.n_valid) {
          float4 bv = b ? *reinterpret_cast<const float4*>(b + c) : make_float4(0.f, 0.f, 0.f, 0.f);
          *reinterpret_cast<float4*>(o + c) = make_float4(acc[i] + bv.x, acc[i + 1] + bv.y, acc[i + 2] + bv.z, acc[i + 3] + bv.w);
        }
      }
    } else {
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        int c = col0 + i;
        if (c < e.n_valid) o[c] = acc[i] + (b ? b[c] : 0.f);
      }
    }
  } else if (EPI == EPI_ELU_C8 || EPI == EPI_DACT_C8) {
    float v[16];
    if (EPI == EPI_DACT_C8) {
      const uint4* a =
          reinterpret_cast<const uint4*>(e.act + rc.model * e.act_ms) + ((long long)(col0 >> 3) * e.act_rcap + e.act_row0 + rc.row);
      uint4 q0 = a[0];
      uint4 q1 = a[e.act_rcap];
      float h[16];
      float h0[8], h1[8];
      unpack_bf16x8(q0, h0);
      unpack_bf16x8(q1, h1);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        h[i] = h0[i];
        h[8 + i] = h1[i];
      }
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        bool ok = rc.valid && (col0 + i) < e.n_valid;
        v[i] = ok ? acc[i] * elu1_grad_from_out(h[i]) : 0.f;
      }
    } else {
      const float* b = e.bias + rc.model * e.bias_ms + col0;
      const float* cb = e.clsb ? e.clsb + rc.model * e.clsb_ms + (long long)rc.cls * e.clsb_ld + col0 : nullptr;
      float bb[16];
#pragma unroll
      for (int i = 0; i < 16; i += 4) {
        float4 t = *reinterpret_cast<const float4*>(b + i);
        if (cb) {
          float4 u = *reinterpret_cast<const float4*>(cb + i);
          t.x += u.x;
          t.y += u.y;
          t.z += u.z;
          t.w += u.w;
        }
        bb[i] = t.x;
        bb[i + 1] = t.y;
        bb[i + 2] = t.z;
        bb[i + 3] = t.w;
      }
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        int c = col0 + i;
        const float x = elu1(acc[i] + bb[i]);
        // column n_valid is the ones column the next layer's dW turns into its bias gradient
        v[i] = !rc.valid ? 0.f : (c < e.n_valid ? x : (c == e.n_valid ? 1.f : 0.f));
      }
    }
    uint4* o = reinterpret_cast<uint4*>(e.out_c8 + rc.model * e.out_c8_ms) +
               ((long long)(col0 >> 3) * e.out_c8_rcap + e.out_c8_row0 + rc.row);
    o[0] = pack_bf16x8(v);
    o[e.out_c8_rcap] = pack_bf16x8(v + 8);
  } else if (EPI == EPI_GRAD) {
    const int k = rc.row;  // input feature (or ones / class column)
    if (k >= e.g_kaug || col0 >= e.g_tab_n) return;  // (weight-gradient tiles need not divide the shadow rows)
    // flat parameter index of column i: weight W[n][k], bias b[n] or class column W[n][kin + j]
    // (tables are warp-uniform: broadcast loads)
    const int4* tw = reinterpret_cast<const int4*>(e.g_tab + (k == e.g_kin ? e.g_tab_n : 0) + col0);
    const int kofs = (k < e.g_kin) ? k : (k == e.g_kin ? 0 : k - 1);
    int idx[16];
#pragma unroll
    for (int i = 0; i < 16; i += 4) {
      const int4 t = tw[i >> 2];
      idx[i] = t.x, idx[i + 1] = t.y, idx[i + 2] = t.z, idx[i + 3] = t.w;
    }
    float* g = e.grad + rc.model * e.grad_ms + kofs;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      if (idx[i] >= 0) {
        if (atomic)
          atomicAdd(g + idx[i], acc[i]);
        else
          g[idx[i]] = acc[i];
      }
    }
  }
}

// One (mu, sigma) element of the decoder-loss epilogue.  Reference math: sigma = softplus(s) + 1e-3
// (src/blocks.py:410-416), log N(t; mu, sigma) (src/blocks.py:230-234) and its gradient towards the two
// pre-activations, scaled by ncoef = -(loss coefficient of the row).  One exponential serves softplus and its
// derivative; divisions are reciprocal-multiplies and the transcendentals the flush-to-zero hardware approximations:
// without .ftz every ex2 / lg2 / rcp carries a denormal-range fix-up (set-predicate + two multiplies), a third of the
// instructions of a kernel that ncu shows issue-bound (65 % issue-active, profiles/r02_experiments.md).
__device__ __forceinline__ float fast_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float fast_lg2(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float fast_rcp(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// two features at a time: the additions, multiplications and fused multiply-adds as packed fp32 pairs (same IEEE
// rounding per element); the transcendentals, comparisons and selects stay scalar
__device__ __forceinline__ float2 decloss_pair(float2 mu, float2 sp, float2 tgt, float ncoef, float2& dmu, float2& dsg) {
  const float LOG2E = 1.4426950408889634f, LN2 = 0.6931471805599453f, HALF_LOG2PI = 0.9189385332046727f;
  const float2 x = mul2(make_float2(fminf(sp.x, 20.f), fminf(sp.y, 20.f)), splat2(LOG2E));
  const float2 ex = make_float2(fast_ex2(x.x), fast_ex2(x.y));
  const float2 one_ex = add2(ex, splat2(1.f));
  const float2 l1p = mul2(make_float2(fast_lg2(one_ex.x), fast_lg2(one_ex.y)), splat2(LN2));
  const float2 tiny = mul2(ex, fma2(splat2(-0.5f), ex, splat2(1.f)));  // log1p(ex) for ex < 1e-3
  const float2 soft = make_float2(ex.x < 1e-3f ? tiny.x : l1p.x, ex.y < 1e-3f ? tiny.y : l1p.y);
  const bool bx = sp.x > 20.f, by = sp.y > 20.f;
  const float2 sg = add2(make_float2(bx ? sp.x : soft.x, by ? sp.y : soft.y), splat2(1e-3f));
  const float2 sgm = mul2(ex, make_float2(fast_rcp(one_ex.x), fast_rcp(one_ex.y)));
  const float2 sig = make_float2(bx ? 1.f : sgm.x, by ? 1.f : sgm.y);  // d softplus / d s
  const float2 inv = make_float2(fast_rcp(sg.x), fast_rcp(sg.y));
  const float2 t = mul2(fma2(mu, splat2(-1.f), tgt), inv);  // (tgt - mu) / sg
  const float2 lg = make_float2(fast_lg2(sg.x), fast_lg2(sg.y));
  const float2 lp = fma2(mul2(splat2(-0.5f), t), t, fma2(splat2(-LN2), lg, splat2(-HALF_LOG2PI)));
  // d CMPL / d mu = -coef (t - mu) / sg^2 ;  d CMPL / d sg = -coef ((t - mu)^2 / sg^3 - 1 / sg)
  const float2 c1 = mul2(splat2(ncoef), inv);
  dmu = mul2(c1, t);
  dsg = mul2(mul2(c1, fma2(t, t, splat2(-1.f))), sig);
  return lp;
}

// Decoder heads: acc_mu / acc_sg are the mu and sigma pre-activations of features
// [f0, f0+16) of one decoder row.  Reference math: src/blocks.py:410-416 (mu, softplus(.)+1e-3)
// and :230-234 (Gaussian log-density with sigma parametrisation).
template <int EPI>
__device__ __forceinline__ void epi_dec_chunk(const EpiParams& e, RowCtx& rc, int f0, int ccol_mu, int ccol_sg,
                                              float (&acc_mu)[16], float (&acc_sg)[16]) {
  const float* b = e.bias + rc.model * e.bias_ms;
  float bmu[16], bsg[16];
#pragma unroll
  for (int i = 0; i < 16; i += 4) {
    const float4 t = *reinterpret_cast<const float4*>(b + ccol_mu + i);
    const float4 u = *reinterpret_cast<const float4*>(b + ccol_sg + i);
    bmu[i] = t.x, bmu[i + 1] = t.y, bmu[i + 2] = t.z, bmu[i + 3] = t.w;
    bsg[i] = u.x, bsg[i + 1] = u.y, bsg[i + 2] = u.z, bsg[i + 3] = u.w;
  }
  if (EPI == EPI_DECOUT) {
    if (!rc.valid) return;
    float* om = e.out_f32 + rc.model * e.out_f32_ms + (long long)(e.out_row0 + rc.row) * e.out_ld;
    float* os = e.out2_f32 + rc.model * e.out_f32_ms + (long long)(e.out_row0 + rc.row) * e.out_ld;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      int f = f0 + i;
      if (f < e.X) {
        om[f] = acc_mu[i] + bmu[i];
        os[f] = softplus20(acc_sg[i] + bsg[i]) + 1e-3f;
      }
    }
    return;
  }
  // EPI_DECLOSS: two halves of 8 features (bias, targets and gradients of 8 features live at a time: the 96-register
  // budget of the 640-thread CTA spilled with all 16).  Chunks that lie entirely inside the real features take the
  // unmasked path; only the last chunk of the last tile masks feature by feature.
  const bool full = f0 + 16 <= e.X;
  const float4* t4 = e.tgt4 + rc.model * e.tgt_ms + (long long)(f0 >> 2) * e.tgt_rcap + (rc.trow < 0 ? 0 : rc.trow);
  uint4* o = reinterpret_cast<uint4*>(e.out_c8 + rc.model * e.out_c8_ms);
  const long long r = e.out_c8_row0 + rc.row;
  const float ncoef = -rc.coef;
  float2 ls2 = make_float2(0.f, 0.f);
#pragma unroll
  for (int hh = 0; hh < 2; ++hh) {
    float tg[8];
#pragma unroll
    for (int i = 0; i < 8; i += 4) {
      float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
      if (rc.trow >= 0 && f0 + hh * 8 + i < e.Xc) t = t4[(long long)(hh * 2 + (i >> 2)) * e.tgt_rcap];
      tg[i] = t.x, tg[i + 1] = t.y, tg[i + 2] = t.z, tg[i + 3] = t.w;
    }
    float dmu[8], dsg[8];
#pragma unroll
    for (int i = 0; i < 8; i += 2) {
      const int j = hh * 8 + i;
      float2 gm, gs;
      const float2 lp = decloss_pair(add2(make_float2(acc_mu[j], acc_mu[j + 1]), make_float2(bmu[j], bmu[j + 1])),
                                     add2(make_float2(acc_sg[j], acc_sg[j + 1]), make_float2(bsg[j], bsg[j + 1])),
                                     make_float2(tg[i], tg[i + 1]), ncoef, gm, gs);
      if (full) {
        ls2 = add2(ls2, lp);
        dmu[i] = gm.x, dmu[i + 1] = gm.y, dsg[i] = gs.x, dsg[i + 1] = gs.y;
      } else {
        const bool ok0 = f0 + j < e.X, ok1 = f0 + j + 1 < e.X;
        ls2 = add2(ls2, make_float2(ok0 ? lp.x : 0.f, ok1 ? lp.y : 0.f));
        dmu[i] = ok0 ? gm.x : 0.f, dmu[i + 1] = ok1 ? gm.y : 0.f;
        dsg[i] = ok0 ? gs.x : 0.f, dsg[i + 1] = ok1 ? gs.y : 0.f;
      }
    }
    if (e.write_dy) {
      o[(long long)((ccol_mu >> 3) + hh) * e.out_c8_rcap + r] = pack_bf16x8(dmu);
      o[(long long)((ccol_sg >> 3) + hh) * e.out_c8_rcap + r] = pack_bf16x8(dsg);
    }
  }
  rc.lsum += ls2.x + ls2.y;  // (rows beyond the dynamic extent: coef = 0 gives zero gradients, epi_end drops their sum)
}

template <int EPI>
__device__ __forceinline__ void epi_end(const EpiParams& e, RowCtx& rc, int tile_n) {
  if (EPI == EPI_DECLOSS) {
    // every row of the tile writes (0 for padding rows) so the reducer can read the padded range
    e.part[rc.model * e.part_ms + (long long)(tile_n * EPI_GROUPS + rc.cg) * e.part_rcap + rc.row] = rc.valid ? rc.lsum : 0.f;
  }
}

// ---------------------------------------------------------------------------------------------
// Tile geometry shared by both kernels
// ---------------------------------------------------------------------------------------------
struct TileInfo {
  int model, tile_m, tile_n, m0, n0;
  int Mrows;  // valid D rows
  int Kc;     // contraction length, multiple of 16
  int kb_begin, kb_end;
  bool active;
};

// tile index -> (model, k-split slice, tile_m, tile_n).  tile = ((model * ksplit + ks) * tiles_mn) + mn
__device__ __forceinline__ TileInfo gemm_tile_info(const GemmProblem& p, int tile) {
  TileInfo t;
  const int tiles_mn = p.tiles_m * p.tiles_n;
  const int mn = tile % tiles_mn;
  const int rest = tile / tiles_mn;
  const int ks = rest % p.ksplit;
  t.model = rest / p.ksplit;
  if (p.mode == GEMM_DW) {
    // weight-gradient tiles: consecutive tiles (running at the same time on neighbouring SMs) take
    // consecutive 128-feature segments of the SAME reference-weight rows
    t.tile_m = mn % p.tiles_m;
    t.tile_n = mn / p.tiles_m;
  } else {
    t.tile_n = mn % p.tiles_n;
    t.tile_m = mn / p.tiles_n;
  }
  t.m0 = t.tile_m * GEMM_BM;
  t.n0 = t.tile_n * p.BN;
  int dyn = p.dyn ? p.dyn[(long long)t.model * p.dyn_stride] : -1;
  if (p.mode == GEMM_DW) {
    t.Mrows = p.M;
    int k = dyn >= 0 ? min(dyn, p.K) : p.K;
    t.Kc = (k + 15) & ~15;
  } else {
    t.Mrows = dyn >= 0 ? min(dyn, p.M) : p.M;
    t.Kc = p.K;
  }
  int nkb = (t.Kc + GEMM_BK - 1) / GEMM_BK;
  int per = (nkb + p.ksplit - 1) / p.ksplit;
  t.kb_begin = min(nkb, ks * per);
  t.kb_end = min(nkb, t.kb_begin + per);
  t.active = t.m0 < t.Mrows && (t.kb_end > t.kb_begin || ks == 0);
  return t;
}

template <int EPI>
__device__ __forceinline__ void run_epilogue_row(const GemmProblem& p, const EpiParams& e, const TileInfo& t, RowCtx& rc,
                                                 uint32_t taddr_row, bool have_acc, bool atomic) {
  epi_begin<EPI>(e, rc);
  if (EPI == EPI_DECLOSS || EPI == EPI_DECOUT) {
    const int hb = p.BN >> 1;
    for (int c = rc.cg * 16; c < hb; c += 16 * EPI_GROUPS) {
      float am[16], as[16];
      if (have_acc) {
        tmem_ld16x2(taddr_row + c, taddr_row + hb + c, am, as);
      } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) am[i] = as[i] = 0.f;
      }
      epi_dec_chunk<EPI>(e, rc, t.tile_n * hb + c, t.n0 + c, t.n0 + hb + c, am, as);
    }
  } else {
    for (int c = rc.cg * 16; c < p.BN; c += 16 * EPI_GROUPS) {
      float acc[16];
      if (have_acc) {
        tmem_ld16(taddr_row + c, acc);
      } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) acc[i] = 0.f;
      }
      epi_chunk<EPI>(e, rc, t.n0 + c, acc, atomic);
    }
  }
  epi_end<EPI>(e, rc, t.tile_n);
}

// ---------------------------------------------------------------------------------------------
// Tensor-core kernel: persistent (one CTA per SM, tiles strided by gridDim.x) and warp-specialised.
//   warp 0        producer: TMA tensor loads of the operand tiles -> shared-memory ring (full/empty mbarriers)
//   warps 1..2    idle
//   warp 3        one elected lane issues tcgen05.mma into one of two TMEM accumulator tiles; owns TMEM
//   warps 4..     epilogue (GEMM_EPI_WARPS): warp w reads TMEM lanes [32(w%4), +32), columns of group (w-4)/4
// The accumulator is double-buffered (acc_full / acc_empty mbarriers), so the epilogue of tile i overlaps the
// mainloop of tile i+1.
// ---------------------------------------------------------------------------------------------
template <int EPI>
__global__ void __launch_bounds__(GEMM_THREADS, 1) gemm_tc_kernel(const GemmProblem p, const EpiParams e,
                                                                 const __grid_constant__ CUtensorMap tmA,
                                                                 const __grid_constant__ CUtensorMap tmB,
                                                                 const __grid_constant__ CUtensorMap tmB2) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(8) uint64_t full_bar[GEMM_MAX_STAGES];
  __shared__ __align__(8) uint64_t empty_bar[GEMM_MAX_STAGES];
  __shared__ __align__(8) uint64_t acc_full[GEMM_ACC_STAGES];
  __shared__ __align__(8) uint64_t acc_empty[GEMM_ACC_STAGES];
  __shared__ uint32_t tmem_base_s;

  TraceScope trace_scope(p.trace, p.trace_id);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int BN = p.BN;
  const int b_stage_bytes = BN * GEMM_BK * 2;
  const int stage_bytes = GEMM_A_STAGE_BYTES + b_stage_bytes;
  uint32_t ncols = 32;
  while ((int)ncols < BN) ncols <<= 1;
  const int total_tiles = p.tiles_m * p.tiles_n * p.ksplit * p.n_models;

  if (threadIdx.x == 0) {
    tma_prefetch_map(&tmA);
    tma_prefetch_map(&tmB);
    tma_prefetch_map(&tmB2);
    for (int s = 0; s < p.nstages; ++s) {
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
    tmem_alloc(&tmem_base_s, GEMM_ACC_STAGES * ncols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;
#ifdef GEMM_PROFILE_WAITS
  const long long ws_cta_t0 = clock64();
#endif

  const bool a_mn = (p.mode == GEMM_DW);
  const bool b_mn = (p.mode != GEMM_NT);

  if (warp == 0) {
    // ===================== producer: TMA tensor loads of operand tiles =====================
    // A chunk8 buffer is the tensor {rcap x 16 B, chunks, models}; a K-major tile is the box
    // {rows, 8 chunks} at (row, k-chunk), an MN-major tile the box {64 contraction rows, MN chunks}
    // at (contraction row, feature chunk).  Boxes are dense in shared memory, which is exactly the
    // [chunk][row][16 B] slab layout of the UMMA descriptors below; rows / chunks beyond the buffer
    // are zero-filled by the TMA unit.  A K-major B tile wider than 128 rows takes two boxes
    // (box extents are limited to 256 elements), multiplied as two N halves.
    // The whole warp walks the ring (uniform control flow), one elected lane issues.
    {
      const uint32_t stage_tx = GEMM_A_STAGE_BYTES + b_stage_bytes;
      const bool b_split = !b_mn && BN > 128;
      uint32_t it = 0;  // k-blocks issued by this CTA so far (ring position)
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const TileInfo t = gemm_tile_info(p, tile);
        if (!t.active) continue;
        for (int kb = t.kb_begin; kb < t.kb_end; ++kb, ++it) {
          const int s = it % p.nstages;
          const uint32_t ph = (it / p.nstages) & 1;
          {
            WS_T0();
            mbar_wait(&empty_bar[s], ph ^ 1, p.dbg, 0xE0000000u | kb);
            if (lane == 0) WS_ADD(WS_PROD_EMPTY);
          }
          uint8_t* As = smem + (size_t)s * stage_bytes;
          uint8_t* Bs = As + GEMM_A_STAGE_BYTES;
          if (elect_one()) {
            mbar_arrive_expect_tx(&full_bar[s], stage_tx);
            if (!a_mn)
              tma_load_3d(As, &tmA, (p.A.row0 + t.m0) * 2, kb * 8, t.model, &full_bar[s]);
            else
              tma_load_3d(As, &tmA, (p.A.row0 + kb * GEMM_BK) * 2, t.m0 >> 3, t.model, &full_bar[s]);
            if (!b_mn) {
              tma_load_3d(Bs, &tmB, (p.B.row0 + t.n0) * 2, kb * 8, t.model, &full_bar[s]);
              if (b_split) tma_load_3d(Bs + 128 * GEMM_BK * 2, &tmB2, (p.B.row0 + t.n0 + 128) * 2, kb * 8, t.model, &full_bar[s]);
            } else {
              tma_load_3d(Bs, &tmB, (p.B.row0 + kb * GEMM_BK) * 2, t.n0 >> 3, t.model, &full_bar[s]);
            }
          }
          __syncwarp();
        }
      }
    }
  } else if (warp == GEMM_MMA_WARP) {
    // ===================== UMMA issuer =====================
    const bool b_split = !b_mn && BN > 128;  // K-major B wider than one TMA box: two N halves
    const int bn0 = b_split ? 128 : BN, bn1 = BN - 128;
    const uint32_t idesc = umma_idesc_bf16(bn0, a_mn ? 1 : 0, b_mn ? 1 : 0);
    const uint32_t idesc1 = b_split ? umma_idesc_bf16(bn1, a_mn ? 1 : 0, 0) : 0u;
    uint32_t a_lbo, a_sbo, a_step, b_lbo, b_sbo, b_step;
    if (!a_mn) {
      a_lbo = GEMM_BM * 16;  // next 8-wide K chunk
      a_sbo = 128;           // next 8 rows
      a_step = 2 * GEMM_BM * 16;
    } else {
      a_lbo = 128;           // next 8 contraction rows
      a_sbo = GEMM_BK * 16;  // next 8-feature MN chunk
      a_step = 16 * 16;
    }
    if (!b_mn) {
      b_lbo = bn0 * 16;
      b_sbo = 128;
      b_step = 2 * bn0 * 16;
    } else {
      b_lbo = 128;
      b_sbo = GEMM_BK * 16;
      b_step = 16 * 16;
    }
    const uint32_t b1_lbo = bn1 * 16, b1_step = 2 * bn1 * 16;
    if (p.desc_variant & 1) {  // bring-up knob: swapped LBO/SBO meaning
      uint32_t x = a_lbo;
      a_lbo = a_sbo;
      a_sbo = x;
      x = b_lbo;
      b_lbo = b_sbo;
      b_sbo = x;
    }
    // One elected lane runs the whole issue loop (the other lanes go to the final barrier).  It is the critical
    // path of every tile, so a k-block is: one barrier wait, the shared-memory address folded into the low
    // descriptor words once, then the MMAs back to back with constant increments (see umma_issue).
    if (elect_one()) {
      const uint64_t a_desc0 = umma_smem_desc(0, a_lbo, a_sbo), b_desc0 = umma_smem_desc(0, b_lbo, b_sbo);
      const uint64_t b1_desc0 = umma_smem_desc(0, b1_lbo, 128);
      const uint32_t a_hi = (uint32_t)(a_desc0 >> 32), b_hi = (uint32_t)(b_desc0 >> 32), b1_hi = (uint32_t)(b1_desc0 >> 32);
      const uint32_t a_lo0 = (uint32_t)a_desc0, b_lo0 = (uint32_t)b_desc0, b1_lo0 = (uint32_t)b1_desc0;
      const uint32_t da = a_step >> 4, db = b_step >> 4, db1 = b1_step >> 4;
      const uint32_t smem0 = smem_u32(smem) >> 4, stage16 = (uint32_t)stage_bytes >> 4;
      uint32_t it = 0, j = 0;  // ring position, active tiles done
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const TileInfo t = gemm_tile_info(p, tile);
        if (!t.active) continue;
        const uint32_t a = j & 1, aph = (j >> 1) & 1;
        {
          WS_T0();
          mbar_wait(&acc_empty[a], aph ^ 1, p.dbg, 0xB0000000u | tile);  // epilogue has drained this accumulator
          WS_ADD(WS_MMA_ACC_EMPTY);
          WS_INC(WS_TILES, 1);
          WS_INC(WS_KBLOCKS, t.kb_end - t.kb_begin);
        }
        tc_fence_after();
        const uint32_t tacc = tmem_base + a * ncols;
        uint32_t s = it % p.nstages, ph = (it / p.nstages) & 1;
        for (int kb = t.kb_begin; kb < t.kb_end; ++kb, ++it) {
          {
            WS_T0();
            mbar_wait(&full_bar[s], ph, p.dbg, 0xF0000000u | kb);
            WS_ADD(WS_MMA_FULL);
          }
          tc_fence_after();
          const int nq = min(GEMM_BK, t.Kc - kb * GEMM_BK) >> 4;
          const uint32_t sa = smem0 + s * stage16;  // (shared address of the stage) >> 4
          const uint32_t alo = a_lo0 + sa, blo = b_lo0 + sa + (GEMM_A_STAGE_BYTES >> 4);
          const uint32_t b1lo = b1_lo0 + sa + ((GEMM_A_STAGE_BYTES + 128 * GEMM_BK * 2) >> 4);
          const uint32_t first = kb > t.kb_begin ? 1u : 0u;
          if (nq == 4 && !b_split) {
            umma_issue(tacc, alo, a_hi, blo, b_hi, idesc, first);
            umma_issue(tacc, alo + da, a_hi, blo + db, b_hi, idesc, 1u);
            umma_issue(tacc, alo + 2 * da, a_hi, blo + 2 * db, b_hi, idesc, 1u);
            umma_issue(tacc, alo + 3 * da, a_hi, blo + 3 * db, b_hi, idesc, 1u);
          } else if (nq == 4) {
            umma_issue(tacc, alo, a_hi, blo, b_hi, idesc, first);
            umma_issue(tacc + 128, alo, a_hi, b1lo, b1_hi, idesc1, first);
            umma_issue(tacc, alo + da, a_hi, blo + db, b_hi, idesc, 1u);
            umma_issue(tacc + 128, alo + da, a_hi, b1lo + db1, b1_hi, idesc1, 1u);
            umma_issue(tacc, alo + 2 * da, a_hi, blo + 2 * db, b_hi, idesc, 1u);
            umma_issue(tacc + 128, alo + 2 * da, a_hi, b1lo + 2 * db1, b1_hi, idesc1, 1u);
            umma_issue(tacc, alo + 3 * da, a_hi, blo + 3 * db, b_hi, idesc, 1u);
            umma_issue(tacc + 128, alo + 3 * da, a_hi, b1lo + 3 * db1, b1_hi, idesc1, 1u);
          } else {
            for (int q = 0; q < nq; ++q) {
              const uint32_t accum = (first | (uint32_t)q) ? 1u : 0u;
              umma_issue(tacc, alo + q * da, a_hi, blo + q * db, b_hi, idesc, accum);
              if (b_split) umma_issue(tacc + 128, alo + q * da, a_hi, b1lo + q * db1, b1_hi, idesc1, accum);
            }
          }
          umma_commit_1t(&empty_bar[s]);  // frees the smem slot once these MMAs retire
          if (++s == (uint32_t)p.nstages) s = 0, ph ^= 1;
        }
        if (t.kb_end > t.kb_begin)
          umma_commit_1t(&acc_full[a]);  // accumulator complete
        else
          mbar_arrive(&acc_full[a]);  // empty contraction: the epilogue uses zeros
        ++j;
      }
    }
    __syncwarp();
  } else if (warp >= GEMM_EPI_WARP0) {
    // ===================== epilogue: TMEM -> registers -> fused math -> HBM =====================
    const int q = warp & 3;                       // TMEM lane quarter this warp may access
    const int cg = (warp - GEMM_EPI_WARP0) >> 2;  // column group
    uint32_t j = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      const TileInfo t = gemm_tile_info(p, tile);
      if (!t.active) continue;
      const uint32_t a = j & 1, aph = (j >> 1) & 1;
      const bool have_acc = t.kb_end > t.kb_begin;
      const uint32_t taddr_row = tmem_base + a * ncols + ((uint32_t)(q * 32) << 16);
      if (lane == 0) {
        WS_T0();
        mbar_wait(&acc_full[a], aph, p.dbg, 0xA0000000u | tile);  // one poller per warp
        if (warp == GEMM_EPI_WARP0) WS_ADD(WS_EPI_ACC_FULL);
      }
      __syncwarp();
      tc_fence_after();
      RowCtx rc;
      rc.model = t.model;
      rc.row = t.m0 + q * 32 + lane;
      rc.cg = cg;
      rc.valid = rc.row < t.Mrows;
      run_epilogue_row<EPI>(p, e, t, rc, taddr_row, have_acc, p.ksplit > 1);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[a]);
      ++j;
    }
  }

#ifdef GEMM_PROFILE_WAITS
  if (lane == 0 && warp == GEMM_EPI_WARP0) WS_INC(WS_EPI_BUSY, clock64() - ws_cta_t0);  // epilogue warp: loop time incl. waits
#endif
  tc_fence_before();
  __syncthreads();
#ifdef GEMM_PROFILE_WAITS
  if (threadIdx.x == 0) WS_INC(WS_CTA_TOTAL, clock64() - ws_cta_t0);
#endif
  if (warp == GEMM_MMA_WARP) tmem_dealloc(tmem_base, GEMM_ACC_STAGES * ncols);
}

// ---------------------------------------------------------------------------------------------
// SIMT validation kernel: same grid, same operands, same epilogues, plain FFMA dot products.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float simt_ldA(const GemmProblem& p, const bf16* A, int mn, int k) {
  long long idx = (p.mode == GEMM_DW) ? c8_index(p.A.row0 + k, mn, p.A.rcap) : c8_index(p.A.row0 + mn, k, p.A.rcap);
  return __bfloat162float(A[idx]);
}
__device__ __forceinline__ float simt_ldB(const GemmProblem& p, const bf16* B, int n, int k) {
  long long idx = (p.mode == GEMM_NT) ? c8_index(p.B.row0 + n, k, p.B.rcap) : c8_index(p.B.row0 + k, n, p.B.rcap);
  return __bfloat162float(B[idx]);
}

template <int EPI>
__global__ void __launch_bounds__(GEMM_SIMT_THREADS) gemm_simt_kernel(const GemmProblem p, const EpiParams e) {
  const TileInfo t = gemm_tile_info(p, blockIdx.x);
  if (!t.active) return;
  const bf16* Ab = p.A.base + t.model * p.A.model_stride;
  const bf16* Bb = p.B.base + t.model * p.B.model_stride;
  RowCtx rc;
  rc.model = t.model;
  rc.row = t.m0 + (threadIdx.x & 127);
  rc.cg = threadIdx.x >> 7;
  rc.valid = rc.row < t.Mrows;
  const int k_lo = t.kb_begin * GEMM_BK;
  const int k_hi = min(t.Kc, t.kb_end * GEMM_BK);
  const bool a_ok = (p.mode == GEMM_DW) ? ((rc.row >> 3) < p.A.nchunks) : (p.A.row0 + rc.row < p.A.rcap);
  epi_begin<EPI>(e, rc);
  auto dot16 = [&](int ncol0, float (&acc)[16]) {
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = 0.f;
    if (!a_ok) return;
    for (int k = k_lo; k < k_hi; ++k) {
      float a = simt_ldA(p, Ab, rc.row, k);
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        int n = ncol0 + i;
        bool b_ok = (p.mode == GEMM_NT) ? (p.B.row0 + n < p.B.rcap) : ((n >> 3) < p.B.nchunks);
        if (b_ok) acc[i] = fmaf(a, simt_ldB(p, Bb, n, k), acc[i]);
      }
    }
  };
  if (EPI == EPI_DECLOSS || EPI == EPI_DECOUT) {
    const int hb = p.BN >> 1;
    for (int c = rc.cg * 16; c < hb; c += 16 * EPI_GROUPS) {
      float am[16], as[16];
      dot16(t.n0 + c, am);
      dot16(t.n0 + hb + c, as);
      epi_dec_chunk<EPI>(e, rc, t.tile_n * hb + c, t.n0 + c, t.n0 + hb + c, am, as);
    }
  } else {
    for (int c = rc.cg * 16; c < p.BN; c += 16 * EPI_GROUPS) {
      float acc[16];
      dot16(t.n0 + c, acc);
      epi_chunk<EPI>(e, rc, t.n0 + c, acc, p.ksplit > 1);
    }
  }
  epi_end<EPI>(e, rc, t.tile_n);
}

// ---------------------------------------------------------------------------------------------
// Host-side launch helper
// ---------------------------------------------------------------------------------------------
enum { GEMM_IMPL_TC = 0, GEMM_IMPL_SIMT = 1 };

inline int gemm_pick_stages(int BN) {
  const int stage = GEMM_A_STAGE_BYTES + BN * GEMM_BK * 2;
  int s = GEMM_SMEM_BUDGET / stage;
  if (s < 2) s = 2;
  if (s > GEMM_MAX_STAGES) s = GEMM_MAX_STAGES;
  return s;
}

inline int gemm_current_device() {
  int dev = 0;
  cudaGetDevice(&dev);
  return (dev >= 0 && dev < 64) ? dev : 0;
}
inline int gemm_num_sms() {
  static int n[64] = {};
  const int dev = gemm_current_device();
  if (n[dev] == 0) {
    if (cudaDeviceGetAttribute(&n[dev], cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n[dev] <= 0) n[dev] = 148;
  }
  return n[dev];
}

// Tensor map of a chunk8 operand buffer: {rcap rows x 16 B (as 2 x 8-byte elements), chunks, models}, box =
// {box_rows, box_chunks, 1}.  Encoded on the host (driver entry point resolved at run time, no libcuda link) and
// cached: a plan launches the same few dozen (buffer, box) combinations every step.
typedef CUresult (*TmapEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline cudaError_t gemm_c8_map(CUtensorMap* out, const GemmOperand& op, int n_models, int box_rows, int box_chunks) {
  static TmapEncodeFn encode = nullptr;
  static std::mutex mu;
  typedef std::tuple<int, const void*, long long, int, int, int, int, int> Key;  // device first: addresses repeat across GPUs
  static std::map<Key, CUtensorMap> cache;
  std::lock_guard<std::mutex> lock(mu);
  if (!encode) {
    void* fp = nullptr;
    cudaDriverEntryPointQueryResult q;
    cudaError_t err = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fp, cudaEnableDefault, &q);
    if (err != cudaSuccess) return err;
    if (!fp || q != cudaDriverEntryPointSuccess) return cudaErrorNotSupported;
    encode = (TmapEncodeFn)fp;
  }
  const Key key(gemm_current_device(), op.base, op.model_stride, op.rcap, op.nchunks, n_models, box_rows, box_chunks);
  auto it = cache.find(key);
  if (it != cache.end()) {
    *out = it->second;
    return cudaSuccess;
  }
  const cuuint64_t chunk_bytes = (cuuint64_t)op.rcap * 16;
  cuuint64_t model_bytes = (cuuint64_t)op.model_stride * 2;
  if (n_models <= 1 || model_bytes == 0) model_bytes = chunk_bytes * (cuuint64_t)op.nchunks;
  if ((model_bytes & 15) || (reinterpret_cast<uintptr_t>(op.base) & 15) || op.rcap < 1 || op.nchunks < 1 || box_rows < 1 ||
      box_rows > 128 || box_chunks < 1 || box_chunks > 256)
    return cudaErrorInvalidValue;
  const cuuint64_t dims[3] = {(cuuint64_t)op.rcap * 2, (cuuint64_t)op.nchunks, (cuuint64_t)(n_models < 1 ? 1 : n_models)};
  const cuuint64_t strides[2] = {chunk_bytes, model_bytes};
  const cuuint32_t box[3] = {(cuuint32_t)box_rows * 2, (cuuint32_t)box_chunks, 1};
  const cuuint32_t es[3] = {1, 1, 1};
  CUtensorMap m;
  CUresult r = encode(&m, CU_TENSOR_MAP_DATA_TYPE_UINT64, 3, const_cast<bf16*>(op.base), dims, strides, box, es,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return cudaErrorInvalidValue;
  if (cache.size() > 4096) cache.clear();  // plans come and go (tests): bound the cache
  cache[key] = m;
  *out = m;
  return cudaSuccess;
}

// The three operand tensor maps of one problem (A tile, B tile, second half of a K-major B tile wider than 128 rows).
inline cudaError_t gemm_make_maps(const GemmProblem& p, int n_models, CUtensorMap* tmA, CUtensorMap* tmB, CUtensorMap* tmB2) {
  const int ens = p.ens > 0 ? p.ens : n_models;
  const bool a_mn = p.mode == GEMM_DW, b_mn = p.mode != GEMM_NT;
  cudaError_t err = a_mn ? gemm_c8_map(tmA, p.A, ens, GEMM_BK, GEMM_BM / 8) : gemm_c8_map(tmA, p.A, ens, GEMM_BM, GEMM_BK / 8);
  if (err != cudaSuccess) return err;
  if (b_mn) {
    err = gemm_c8_map(tmB, p.B, ens, GEMM_BK, p.BN / 8);
    *tmB2 = *tmB;
  } else {
    err = gemm_c8_map(tmB, p.B, ens, p.BN > 128 ? 128 : p.BN, GEMM_BK / 8);
    if (err == cudaSuccess && p.BN > 128) err = gemm_c8_map(tmB2, p.B, ens, p.BN - 128, GEMM_BK / 8);
    if (p.BN <= 128) *tmB2 = *tmB;
  }
  return err;
}

template <int EPI>
inline cudaError_t gemm_launch_t(GemmProblem p, const EpiParams& e, int n_models, int impl, cudaStream_t st) {
  p.n_models = n_models;
  const int total = p.tiles_n * p.tiles_m * p.ksplit * n_models;
  if (impl == GEMM_IMPL_SIMT) {
    gemm_simt_kernel<EPI><<<total, GEMM_SIMT_THREADS, 0, st>>>(p, e);
    return cudaGetLastError();
  }
  p.nstages = gemm_pick_stages(p.BN);
  size_t smem = (size_t)p.nstages * (GEMM_A_STAGE_BYTES + p.BN * GEMM_BK * 2);
  // (function attributes are per device: one process may drive several GPUs)
  static bool attr_set[64] = {};
  const int dev = gemm_current_device();
  if (!attr_set[dev]) {
    cudaError_t err =
        cudaFuncSetAttribute(gemm_tc_kernel<EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BUDGET + 4096);
    if (err != cudaSuccess) return err;
    attr_set[dev] = true;
  }
  // operand tensor maps (see the producer warp of gemm_tc_kernel)
  CUtensorMap tmA, tmB, tmB2;
  cudaError_t err = gemm_make_maps(p, n_models, &tmA, &tmB, &tmB2);
  if (err != cudaSuccess) return err;
  int grid = total < gemm_num_sms() ? total : gemm_num_sms();  // persistent: one CTA per SM
  if (p.max_ctas > 0 && grid > p.max_ctas) grid = p.max_ctas;
  return launch_k(gemm_tc_kernel<EPI>, dim3(grid), dim3(GEMM_THREADS), smem, st, p, e, tmA, tmB, tmB2);
}

inline cudaError_t gemm_launch(int epi, const GemmProblem& p, const EpiParams& e, int n_models, int impl,
                               cudaStream_t st) {
  switch (epi) {
    case EPI_STORE_F32: return gemm_launch_t<EPI_STORE_F32>(p, e, n_models, impl, st);
    case EPI_ELU_C8: return gemm_launch_t<EPI_ELU_C8>(p, e, n_models, impl, st);
    case EPI_DACT_C8: return gemm_launch_t<EPI_DACT_C8>(p, e, n_models, impl, st);
    case EPI_GRAD: return gemm_launch_t<EPI_GRAD>(p, e, n_models, impl, st);
    case EPI_DECLOSS: return gemm_launch_t<EPI_DECLOSS>(p, e, n_models, impl, st);
    case EPI_DECOUT: return gemm_launch_t<EPI_DECOUT>(p, e, n_models, impl, st);
  }
  return cudaErrorInvalidValue;
}

}  // namespace drvae
