// Row-wise kernels of the step: everything between the GEMMs that is local to one minibatch row
// (or one (row, class) evaluation): row-group bookkeeping, input noise, reparameterised sampling,
// analytic KL with free bits, the y classifier, and the assembly of d(loss)/d(pre-activation)
// rows that feed the backward GEMMs.  One warp per row; lane f handles features f, f+32, ...
//
// Reference math (file:line in /root/reference/src):
//   sampling            blocks.py:170-174          z = eps * exp(0.5 logvar) + mu
//   KL(q||p) per row    blocks.py:180-182
//   free bits           DGMMixin.py:68-75          max(KL_row, kl_min)
//   classifier          blocks.py:456-480          clamp(softmax(.), 1e-10, 1-1e-10), log-lik, KL to prior
//   p(z2|z1)            blocks.py:349-361          mu = z + z W^T + b,  logvar = lin(z) - 2
//   group logic         DrVAE.py:367-543, PVAE.py:265-409, VFAE.py:268-401
#pragma once

#include "plan.h"

namespace drvae {

constexpr int ROW_WARPS = 8;            // warps per block in the row kernels
constexpr int ROW_THREADS = ROW_WARPS * 32;
constexpr int PAD_ROWS = 128;           // rows of zero padding kept after the valid rows of a GEMM operand
constexpr int PAD_WARPS = 16;           // extra "pad duty" warps per launch, each zeroing PAD_ROWS / PAD_WARPS rows

// Resident blocks per SM the row kernels are compiled for (register cap = 65536 / (256 x blocks)).  Measured on the
// 32-model step (profiles/r02_experiments.md): one wave of rows matters more than spill-free code for the kernels that
// have one warp per minibatch row.
#ifndef ROW_LB_SAMPLE
#define ROW_LB_SAMPLE 4
#endif
#ifndef ROW_LB_TPOST
#define ROW_LB_TPOST 5
#endif
#ifndef ROW_LB_TBACK
#define ROW_LB_TBACK 4
#endif
#ifndef ROW_LB_QBACK
#define ROW_LB_QBACK 4
#endif
#ifndef ROW_LB_EVAL
#define ROW_LB_EVAL 4
#endif

__device__ __forceinline__ void st_c8(bf16* base, int rcap, int row, int f, float v) {
  base[c8_index(row, f, rcap)] = __float2bfloat16_rn(v);
}
__device__ __forceinline__ void zero_c8_row(const C8Buf& b, int model, int row, int lane) {
  uint4* p = reinterpret_cast<uint4*>(b.at(model));
  const uint4 z = make_uint4(0, 0, 0, 0);
  for (int c = lane; c < (b.fcap >> 3); c += 32) p[(long long)c * b.rcap + row] = z;
}
__device__ __forceinline__ int pad128(int n) { return (n + 127) & ~127; }
// zero the columns of a (d mu | d logvar) gradient row that hold neither half: [Z, Zs) and [Zs + Z, fcap)
__device__ __forceinline__ void zero_c8_gaps(const C8Buf& b, bf16* base, int row, int Z, int Zs, int lane) {
  for (int f = Z + lane; f < Zs; f += 32) st_c8(base, b.rcap, row, f, 0.f);
  for (int f = Zs + Z + lane; f < b.fcap; f += 32) st_c8(base, b.rcap, row, f, 0.f);
}

// ---------------------------------------------------------------------------------------------
// rowmap: split the minibatch into the reference's row groups without moving rows.
// The reference gathers LS / US / LP / UP groups (DrVAE.py:565-608); here every row keeps its
// place and we only record, per row, its pair index, its evaluation slots for _fprop
// (1 for a labeled row, dim_y for an unlabeled one) and the batch-level normalisers.
// ---------------------------------------------------------------------------------------------
constexpr int ROWMAP_THREADS = 1024;

// exclusive prefix sum of one int per thread over the block (warp shuffles + one smem pass); returns the block total in `total`
__device__ __forceinline__ int block_exclusive_scan(int x, int* warp_tot, int& total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int incl = x;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += y;
  }
  if (lane == 31) warp_tot[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int w = lane < nw ? warp_tot[lane] : 0;
    int wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, wi, o);
      if (lane >= o) wi += y;
    }
    warp_tot[lane] = wi - w;  // exclusive prefix of the warp totals
    if (lane == 31) warp_tot[32] = wi;
  }
  __syncthreads();
  const int res = warp_tot[warp] + incl - x;
  total = warp_tot[32];
  __syncthreads();
  return res;
}

__global__ void __launch_bounds__(ROWMAP_THREADS) rowmap_kernel(DevView v) {
  TraceScope trace_scope(v.trace, v.trace_id);
  const int m = blockIdx.x, t = threadIdx.x, N = v.N;
  __shared__ int s_tot[33];
  const int* hx = v.has_pair ? v.has_x2.at(m) : nullptr;
  const int* hy = (v.has_clf && v.has_y.p) ? v.has_y.at(m) : nullptr;
  const int* yy = (v.has_clf && v.y.p) ? v.y.at(m) : nullptr;
  const int* ri = v.row_index.p ? v.row_index.at(m) : nullptr;  // batch row -> dataset row (device-resident dataset)
  const int seg = (N + ROWMAP_THREADS - 1) / ROWMAP_THREADS;
  const int i0 = min(N, t * seg), i1 = min(N, i0 + seg);
  int np = 0, ne = 0, nl = 0;
  for (int i = i0; i < i1; ++i) {
    const int di = ri ? ri[i] : i;
    const bool pr = hx && hx[di] != 0;
    const bool lb = hy && hy[di] != 0;
    np += pr;
    nl += lb;
    ne += v.has_fprop ? (lb ? 1 : v.Y) : 0;
  }
  int Np, Fl, Nlab;
  int p = block_exclusive_scan(np, s_tot, Np);
  int e = block_exclusive_scan(ne, s_tot, Fl);
  (void)block_exclusive_scan(nl, s_tot, Nlab);
  if (t == 0) {
    int* cnt = v.counts.at(m);
    cnt[CNT_N] = N;
    cnt[CNT_NP] = Np;
    cnt[CNT_NLAB] = Nlab;
    cnt[CNT_R0] = N + Np;
    cnt[CNT_LN] = v.L * N;
    cnt[CNT_LNP] = v.L * Np;
    cnt[CNT_RD] = v.L * (N + 2 * Np);
    cnt[CNT_FL] = Fl;
    cnt[CNT_F] = v.L * Fl;
    const float gN = v.dyn->s.gN > 0 ? v.dyn->s.gN : N;
    const float gNp = fmaxf(1.f, v.dyn->s.gN > 0 ? v.dyn->s.gNp : Np);
    const float gNl = fmaxf(1.f, v.dyn->s.gN > 0 ? v.dyn->s.gNlab : Nlab);
    const float Lf = v.L;
    float* cf = v.coefs.at(m);
    cf[COEF_RECL] = 1.f / (Lf * gN);
    cf[COEF_PERT] = v.dyn->s.beta_pert * v.member(m).pertloss_rate / (Lf * gNp);
    cf[COEF_KLZ2] = v.dyn->s.beta_pert * v.member(m).kl_qz2pz2_rate / (Lf * gN);
    cf[COEF_KLD] = 1.f / (Lf * gN);
    cf[COEF_YL] = v.member(m).yloss_rate / (Lf * gNl);
    cf[COEF_INV_N] = 1.f / gN;
    cf[COEF_PERT_PLAIN] = 1.f / (Lf * gNp);
    cf[COEF_YL_PLAIN] = 1.f / (Lf * gNl);
  }
  int* pair_of = v.pair_of.at(m);
  int* row_of_pair = v.row_of_pair.at(m);
  int* ebase = v.ebase.at(m);
  int* lab = v.lab.at(m);
  int* ycls = v.ycls.at(m);
  int* e_row = v.e_row.at(m);
  int* e_jj = v.e_jj.at(m);
  for (int i = i0; i < i1; ++i) {
    const int di = ri ? ri[i] : i;
    const bool pr = hx && hx[di] != 0;
    const bool lb = hy && hy[di] != 0;
    int yi = yy ? yy[di] : 0;
    yi = min(max(yi, 0), v.Y - 1);
    pair_of[i] = pr ? p : -1;
    if (pr) row_of_pair[p++] = i;
    lab[i] = lb;
    ycls[i] = yi;
    ebase[i] = e;
    if (v.has_fprop) {
      const int c = lb ? 1 : v.Y;
      for (int jj = 0; jj < c; ++jj) {
        e_row[e + jj] = i;
        e_jj[e + jj] = jj;
      }
      e += c;
    }
  }
  __syncthreads();
  if (v.has_fprop) {
    int* full = v.e_cls_full.at(m);
    for (int k = t; k < v.L * Fl; k += ROWMAP_THREADS) {
      const int el = k % Fl;
      const int i = e_row[el];
      full[k] = lab[i] ? ycls[i] : e_jj[el];
    }
  }
}

// ---------------------------------------------------------------------------------------------
// prep: encoder input rows.  Row r < N is x1[r]; row N + p is x2 of the p-th pair.  With
// --train-w-noise the noisy row is ALSO the reconstruction target (DrVAE.py:404-417 adds the
// noise in place), so the fp32 target copy is written from the same value.
// Reads are coalesced along features, writes along rows (the chunk8 bf16 GEMM operand with its
// ones column at feature X, and the chunk4 fp32 target the decoder epilogue reads), through a
// shared-memory transpose of 32 rows x 256 features.
// grid (R0cap / 32, ceil(Xc / 256), n_models), block 256
// ---------------------------------------------------------------------------------------------
constexpr int PREP_ROWS = 32;
constexpr int PREP_THREADS = 256;
constexpr int PREP_SLAB = 256;

__global__ void __launch_bounds__(PREP_THREADS) prep_kernel(DevView v) {
  TraceScope trace_scope(v.trace, v.trace_id);
  __shared__ float tile[PREP_ROWS][PREP_SLAB + 1];
  const int m = blockIdx.z, r0 = blockIdx.x * PREP_ROWS;
  const int* cnt = v.counts.at(m);
  const int N = cnt[CNT_N], R0 = cnt[CNT_R0];
  if (r0 >= pad128(R0)) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool noisy = v.dyn->s.training && v.dyn->s.add_noise;
  uint4* ain = reinterpret_cast<uint4*>(v.Ain.at(m));
  float4* tg = v.tgt4.at(m);
  {
    const int f0 = blockIdx.y * PREP_SLAB;
    const int fw = min(PREP_SLAB, v.Xc - f0);  // multiple of 16
    // phase 1: one warp per row, each lane 4 consecutive features (one Philox quad) at a time
    for (int rl = warp; rl < PREP_ROWS; rl += PREP_THREADS / 32) {
      const int r = r0 + rl;
      const float* src = nullptr;
      const float* eps = nullptr;
      int seg = 0, nrow = 0;  // noise keys: draw kind and row inside this model's minibatch
      if (r < N) {
        nrow = r;
        src = v.x1.at(m) + (long long)(v.row_index.p ? v.row_index.at(m)[r] : r) * v.X;
        eps = v.eps_x1.at(m) + (long long)r * v.X;
      } else if (r < R0) {
        nrow = v.row_of_pair.at(m)[r - N];
        seg = 1;
        src = v.x2.at(m) + (long long)(v.row_index.p ? v.row_index.at(m)[nrow] : nrow) * v.X;
        eps = v.eps_x2.at(m) + (long long)nrow * v.X;
      }
      for (int qd = lane; qd < (fw >> 2); qd += 32) {
        const int f = f0 + qd * 4;
        float x[4] = {0.f, 0.f, 0.f, 0.f};
        if (src && f < v.X) {
          float z[4] = {0.f, 0.f, 0.f, 0.f};
          if (noisy && v.own_noise) philox_normal4(v.dyn->noise_seed, v.dyn->noise_step, m, seg, 0, (unsigned long long)(v.dyn->row_offset + nrow), f >> 2, z);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            if (f + k < v.X) {
              x[k] = src[f + k];
              if (noisy) x[k] += v.member(m).noise_std * (v.own_noise ? z[k] : eps[f + k]);
            }
          }
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) tile[rl][qd * 4 + k] = x[k];
      }
    }
    __syncthreads();
    // phase 2: lanes along rows, one 8-feature chunk per (warp, iteration)
    const int r = r0 + lane;
    for (int c = warp; c < (fw >> 3); c += PREP_THREADS / 32) {
      float a[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) a[k] = tile[lane][c * 8 + k];
      const int fc = f0 + c * 8;
      tg[(long long)(fc >> 2) * v.R0cap + r] = make_float4(a[0], a[1], a[2], a[3]);
      tg[(long long)((fc >> 2) + 1) * v.R0cap + r] = make_float4(a[4], a[5], a[6], a[7]);
#pragma unroll
      for (int k = 0; k < 8; ++k)
        if (fc + k == v.X && r < R0) a[k] = 1.f;  // ones column (bias gradient of the first layer)
      ain[(long long)(fc >> 3) * v.Ain.rcap + r] = pack_bf16x8(a);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// classifier q(y | u): u = [z1, z2f - z1] (DrVAE) or z1 (VFAE).  Warp-cooperative, fp32.
// ---------------------------------------------------------------------------------------------
// The classifier's output stage: acc[j] holds lane-partial logits (bias not yet added).  Shuffle-tree sum, softmax,
// clamp (blocks.py:462), then q(y|.) and the row's label terms.
__device__ __forceinline__ void classifier_tail(const DevView& v, int m, int r, int i, int lane, float (&acc)[MAXY]) {
  const float* bc = v.params.at(m) + v.clf_b_off;
  float mx = -INFINITY;
#pragma unroll
  for (int j = 0; j < MAXY; ++j) {
    if (j < v.Y) {
      acc[j] = warp_sum(acc[j]) + bc[j];
      mx = fmaxf(mx, acc[j]);
    }
  }
  float den = 0.f;
#pragma unroll
  for (int j = 0; j < MAXY; ++j) {
    if (j < v.Y) {
      acc[j] = expf(acc[j] - mx);
      den += acc[j];
    }
  }
  float yl = 0.f, ycat = 0.f;
  const bool lb = v.lab.at(m)[i] != 0;
  const int yi = v.ycls.at(m)[i];
#pragma unroll
  for (int j = 0; j < MAXY; ++j) {
    if (j < v.Y) {
      float q = acc[j] / den;
      q = fminf(fmaxf(q, 1e-10f), 1.f - 1e-10f);
      if (lane == 0) v.QY.at(m)[(long long)r * v.Y + j] = q;
      const float lq = logf(q);
      if (lb) {
        if (j == yi) yl = lq;
      } else {
        ycat += -q * (v.member(m).log_prior[j] - lq);
      }
    }
  }
  if (lane == 0) {
    v.yl_row.at(m)[r] = yl;
    v.ycat_row.at(m)[r] = ycat;
  }
}

__device__ __forceinline__ void classifier_row(const DevView& v, int m, int r, int i, int lane) {
  const float* Wc = v.clf_w.at(m);
  const float* z1 = v.Z1f.at(m) + (long long)r * v.Z;
  const float* z2f = (v.clf_in > v.Z) ? v.Z2Ff.at(m) + (long long)r * v.Z : nullptr;
  float acc[MAXY];
#pragma unroll
  for (int j = 0; j < MAXY; ++j) acc[j] = 0.f;
  for (int f = lane; f < v.Z; f += 32) {
    const float a = z1[f];
    const float d = z2f ? z2f[f] - a : 0.f;
#pragma unroll
    for (int j = 0; j < MAXY; ++j) {
      if (j < v.Y) {
        acc[j] = fmaf(Wc[j * v.clf_ld + f], a, acc[j]);
        if (z2f) acc[j] = fmaf(Wc[j * v.clf_ld + v.Z + f], d, acc[j]);
      }
    }
  }
  classifier_tail(v, m, r, i, lane, acc);
}

// The same classifier with its input taken from registers: feature f = lane + 32 k of z1 (and of z2f when the
// classifier sees [z1, z2f - z1]).  Same accumulation order as classifier_row (k ascending per lane, then the shuffle
// tree), so both give bit-identical results; this form has no global round trip for the row the caller has just
// computed and issues all weight loads back to back.
template <int J>
__device__ __forceinline__ void classifier_row_regs(const DevView& v, int m, int r, int i, int lane, const float (&z1)[J],
                                                    const float (&z2f)[J], bool two) {
  const float* Wc = v.clf_w.at(m);
  float acc[MAXY];
#pragma unroll
  for (int j = 0; j < MAXY; ++j) acc[j] = 0.f;
#pragma unroll
  for (int k = 0; k < J; ++k) {
    const int f = lane + 32 * k;
    if (f < v.Z) {
      const float a = z1[k];
      const float d = two ? z2f[k] - a : 0.f;
#pragma unroll
      for (int j = 0; j < MAXY; ++j) {
        if (j < v.Y) {
          acc[j] = fmaf(Wc[j * v.clf_ld + f], a, acc[j]);
          if (two) acc[j] = fmaf(Wc[j * v.clf_ld + v.Z + f], d, acc[j]);
        }
      }
    }
  }
  classifier_tail(v, m, r, i, lane, acc);
}

// The classifier with hidden layers: linear_p (fp32 weights) over the last hidden activation of stacked row r (bf16
// chunk8, ClfView::pin features); lane l takes the 8-feature chunks l, l + 32, ...
__device__ __forceinline__ void classifier_row_h(const DevView& v, int m, int r, int i, int lane) {
  const ClfView& cv = *v.clf;
  const float* Wc = v.clf_w.at(m);
  const uint4* hp = reinterpret_cast<const uint4*>(cv.H.at(m)) + r;
  float acc[MAXY];
#pragma unroll
  for (int j = 0; j < MAXY; ++j) acc[j] = 0.f;
  for (int c = lane; c < (cv.pin + 7) >> 3; c += 32) {
    float h[8];
    unpack_bf16x8(hp[(long long)c * cv.H.rcap], h);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int f = 8 * c + e;
      if (f < cv.pin) {
#pragma unroll
        for (int j = 0; j < MAXY; ++j)
          if (j < v.Y) acc[j] = fmaf(Wc[j * v.clf_ld + f], h[e], acc[j]);
      }
    }
  }
  classifier_tail(v, m, r, i, lane, acc);
}

__device__ __forceinline__ float kl_prior_term(float mu, float lv) { return 0.5f * (-lv - 1.f + mu * mu + expf(lv)); }
__device__ __forceinline__ float kl_term(float muq, float lvq, float mup, float lvp) {
  const float d = muq - mup;
  return 0.5f * (lvp - lvq - 1.f + (d * d + expf(lvq)) * expf(-lvp));
}

// ---------------------------------------------------------------------------------------------
// sample_q1: after the encoder heads.  Draw z1 (and z2 — from q(z1|x1), as the reference does,
// DrVAE.py:427) for every MC sample and scatter them to the stacked decoder rows.
// grid (ceil((N + PAD_WARPS) / ROW_WARPS), n_models)
// ---------------------------------------------------------------------------------------------
// J: feature slots per lane held in registers (latent dim <= 32 J); 4 covers the README's 100-dim latents within the
// 48-register budget of 5 blocks per SM, MAXJ is the general case
template <int J>
__device__ __forceinline__ void sample_q1_row(const DevView& v, const int m, const int i, const int lane) {
  const int* cnt = v.counts.at(m);
  const int N = cnt[CNT_N], Np = cnt[CNT_NP], LN = cnt[CNT_LN], Fl = cnt[CNT_FL], F = cnt[CNT_F], Rd = cnt[CNT_RD];
  if (i >= N) {
    const int j = i - N;  // pad duty
    if (j < PAD_WARPS) {
      for (int jj = j; jj < PAD_ROWS; jj += PAD_WARPS) {
        if (v.has_fprop && F + jj < pad128(F)) zero_c8_row(v.Z1e, m, F + jj, lane);
        if (!v.has_T && Rd + jj < pad128(Rd)) zero_c8_row(v.Zdec, m, Rd + jj, lane);
      }
    }
    return;
  }
  const float* q = v.Q.at(m) + (long long)i * 2 * v.Zs;
  const int p = v.pair_of.at(m)[i];
  const int eb = v.has_fprop ? v.ebase.at(m)[i] : 0;
  const int ecnt = v.has_fprop ? (v.lab.at(m)[i] ? 1 : v.Y) : 0;
  bf16* zdec = v.Zdec.at(m);
  bf16* z1e = v.has_fprop ? v.Z1e.at(m) : nullptr;
  const int ycl = v.has_fprop ? v.ycls.at(m)[i] : 0;
  // q(z1|x1) statistics of this row, staged in registers: feature f = lane + 32 k
  float mu[J], sd[J];
#pragma unroll
  for (int k = 0; k < J; ++k) {
    const int f = lane + 32 * k;
    mu[k] = f < v.Z ? q[f] : 0.f;
    sd[k] = f < v.Z ? expf(0.5f * q[v.Zs + f]) : 0.f;
  }
  for (int l = 0; l < v.L; ++l) {
    const int r = l * N + i;
    const float* e1 = v.eps_z1.at(m) + ((long long)l * v.Ncap + i) * v.Z;
    const float* e2 = v.eps_z2.at(m) + ((long long)l * v.Ncap + i) * v.Z;
    float n1[J], n2[J];
#pragma unroll
    for (int k = 0; k < J; ++k) {  // all noise loads of this sample before the first store
      const int f = lane + 32 * k;
      n1[k] = f < v.Z ? e1[f] : 0.f;
      n2[k] = (f < v.Z && p >= 0) ? e2[f] : 0.f;
    }
#pragma unroll
    for (int k = 0; k < J; ++k) {
      const int f = lane + 32 * k;
      if (f >= v.Zc) continue;
      // feature Z is the ones column (bias gradients); features Z+1+j are the one-hot class
      // columns of the [z1, onehot(y)] input of q(z_top | z1, y)
      float z = (f == v.Z) ? 1.f : 0.f, z2 = z;
      if (f < v.Z) {
        z = mu[k] + sd[k] * n1[k];
        v.Z1f.at(m)[(long long)r * v.Z + f] = z;
        if (p >= 0) z2 = mu[k] + sd[k] * n2[k];
      }
      st_c8(zdec, v.Zdec.rcap, r, f, z);
      if (p >= 0) st_c8(zdec, v.Zdec.rcap, LN + l * Np + p, f, z2);
      for (int jj = 0; jj < ecnt; ++jj) {
        const int cls = ecnt == 1 ? ycl : jj;
        st_c8(z1e, v.Z1e.rcap, l * Fl + eb + jj, f, (f == v.Z + 1 + cls) ? 1.f : z);
      }
      n1[k] = z;  // (kept for the classifier below)
    }
    // features past the register slots (dim_z1 near 32 J): only constant columns, the ones column and the one-hot
    // class columns, can lie there
    for (int f = 32 * J + lane; f < v.Zc; f += 32) {
      const float z = (f == v.Z) ? 1.f : 0.f;
      st_c8(zdec, v.Zdec.rcap, r, f, z);
      if (p >= 0) st_c8(zdec, v.Zdec.rcap, LN + l * Np + p, f, z);
      for (int jj = 0; jj < ecnt; ++jj) {
        const int cls = ecnt == 1 ? ycl : jj;
        st_c8(z1e, v.Z1e.rcap, l * Fl + eb + jj, f, (f == v.Z + 1 + cls) ? 1.f : z);
      }
    }
    if (v.has_clf && !v.has_T && !v.clf) classifier_row_regs<J>(v, m, r, i, lane, n1, n1, false);
  }
  if (v.kind == KIND_PVAE) {  // KL(q1 || N(0,I)) and KL(q2 || N(0,I)) with free bits (PVAE.py:330-372)
    float k1 = 0.f, k2 = 0.f;
    const float* q2 = p >= 0 ? v.Q.at(m) + (long long)(N + p) * 2 * v.Zs : nullptr;
    for (int f = lane; f < v.Z; f += 32) {
      k1 += kl_prior_term(q[f], q[v.Zs + f]);
      if (q2) k2 += kl_prior_term(q2[f], q2[v.Zs + f]);
    }
    k1 = warp_sum(k1);
    k2 = warp_sum(k2);
    if (lane == 0) {
      v.klq_row.at(m)[i] = fmaxf(k1, v.dyn->s.kl_min);
      if (p >= 0) v.klq_row.at(m)[N + p] = fmaxf(k2, v.dyn->s.kl_min);
    }
  }
}

template <int J>
__global__ void __launch_bounds__(ROW_THREADS, ROW_LB_SAMPLE) sample_q1_kernel(DevView v) {
  TraceScope trace_scope(v.trace, v.trace_id);
  sample_q1_row<J>(v, blockIdx.y, blockIdx.x * ROW_WARPS + (threadIdx.x >> 5), threadIdx.x & 31);
}

// ---------------------------------------------------------------------------------------------
// T_post: after the p(z2|z1) GEMM.  Residual mean, sample z2f, KL(q(z2|x2) || p(z2|z1)) with free
// bits for pair rows, and the classifier.
// ---------------------------------------------------------------------------------------------
template <int J>
__device__ __forceinline__ void T_post_row(const DevView& v, const int m, const int i, const int lane) {
  const int* cnt = v.counts.at(m);
  const int N = cnt[CNT_N], Np = cnt[CNT_NP], LN = cnt[CNT_LN], LNp = cnt[CNT_LNP], Rd = cnt[CNT_RD];
  if (i >= N) {
    const int j = i - N;
    if (j < PAD_WARPS)
      for (int jj = j; jj < PAD_ROWS; jj += PAD_WARPS)
        if (Rd + jj < pad128(Rd)) zero_c8_row(v.Zdec, m, Rd + jj, lane);
    return;
  }
  const int p = v.pair_of.at(m)[i];
  const float* q2 = p >= 0 ? v.Q.at(m) + (long long)(N + p) * 2 * v.Zs : nullptr;
  bf16* zdec = v.Zdec.at(m);
  for (int l = 0; l < v.L; ++l) {
    const int r = l * N + i;
    float* pt = v.PT.at(m) + (long long)r * 2 * v.Zs;
    const float* z1 = v.Z1f.at(m) + (long long)r * v.Z;
    const float* ef = v.eps_z2f.at(m) + ((long long)l * v.Ncap + i) * v.Z;
    float kl = 0.f;
    float a_pmu[J], a_plv[J], a_z1[J], a_ef[J], a_q2m[J], a_q2l[J];
#pragma unroll
    for (int k = 0; k < J; ++k) {  // every load of this sample before the first store
      const int f = lane + 32 * k;
      const bool in = f < v.Z;
      a_pmu[k] = in ? pt[f] : 0.f;
      a_plv[k] = in ? pt[v.Zs + f] : 0.f;
      a_z1[k] = in ? z1[f] : 0.f;
      a_ef[k] = in ? ef[f] : 0.f;
      a_q2m[k] = (in && q2) ? q2[f] : 0.f;
      a_q2l[k] = (in && q2) ? q2[v.Zs + f] : 0.f;
    }
#pragma unroll
    for (int k = 0; k < J; ++k) {
      const int f = lane + 32 * k;
      if (f >= v.Zc) continue;
      float z2f = (f == v.Z) ? 1.f : 0.f;  // ones column
      if (f < v.Z) {
        const float pmu = a_pmu[k] + a_z1[k];
        const float plv = a_plv[k];
        pt[f] = pmu;
        z2f = pmu + expf(0.5f * plv) * a_ef[k];
        v.Z2Ff.at(m)[(long long)r * v.Z + f] = z2f;
        if (q2) kl += kl_term(a_q2m[k], a_q2l[k], pmu, plv);
      }
      if (p >= 0) st_c8(zdec, v.Zdec.rcap, LN + LNp + l * Np + p, f, z2f);
      a_ef[k] = z2f;  // (kept for the classifier below)
    }

    if (p >= 0)  // constant columns past the register slots (see sample_q1_row)
      for (int f = 32 * J + lane; f < v.Zc; f += 32) st_c8(zdec, v.Zdec.rcap, LN + LNp + l * Np + p, f, (f == v.Z) ? 1.f : 0.f);
    kl = warp_sum(kl);
    if (lane == 0) v.klz2_row.at(m)[r] = q2 ? fmaxf(kl, v.dyn->s.kl_min) : 0.f;
    if (v.has_clf && !v.clf) classifier_row_regs<J>(v, m, r, i, lane, a_z1, a_ef, v.clf_in > v.Z);
  }
}

template <int J>
__global__ void __launch_bounds__(ROW_THREADS, ROW_LB_TPOST) T_post_kernel(DevView v) {
  TraceScope trace_scope(v.trace, v.trace_id);
  T_post_row<J>(v, blockIdx.y, blockIdx.x * ROW_WARPS + (threadIdx.x >> 5), threadIdx.x & 31);
}

// ---------------------------------------------------------------------------------------------
// clf_fwd: the output layer linear_p of a classifier with hidden layers (DevView::clf), one warp per stacked row
// r = l * N + i, after the hidden layers' GEMMs.  Only the label-dependent branch and the backward need q(y|.), the
// decoder does not: it runs on the side stream, and sample_q1 / T_post stay as without hidden layers.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void clf_fwd_row(const DevView& v, const int m, const int r, const int lane) {
  const int* cnt = v.counts.at(m);
  const int N = cnt[CNT_N], LN = cnt[CNT_LN];
  if (r >= LN) return;
  classifier_row_h(v, m, r, r % N, lane);
}

__global__ void __launch_bounds__(ROW_THREADS) clf_fwd_kernel(DevView v) {
  TraceScope trace_scope(v.trace, v.trace_id);
  clf_fwd_row(v, blockIdx.y, blockIdx.x * ROW_WARPS + (threadIdx.x >> 5), threadIdx.x & 31);
}

// clf_u (DrVAE, classifier hidden layers): the first hidden GEMM's operand u = [z1 | z2f - z1 | 1] of stacked row r, as
// bf16 chunk8, from the fp32 samples sample_q1 / T_post have stored.  Runs next to the classifier's GEMMs, off the
// main chain (T_post itself is the same as without hidden layers).
__device__ __forceinline__ void clf_u_row(const DevView& v, const int m, const int r, const int lane) {
  if (r >= v.counts.at(m)[CNT_LN]) return;
  const C8Buf& U = v.clf->U;
  bf16* u = U.at(m);
  const float* z1 = v.Z1f.at(m) + (long long)r * v.Z;
  const float* z2f = v.Z2Ff.at(m) + (long long)r * v.Z;
  for (int f = lane; f < U.fcap; f += 32) {
    float x = (f == 2 * v.Z) ? 1.f : 0.f;
    if (f < v.Z)
      x = z1[f];
    else if (f < 2 * v.Z)
      x = z2f[f - v.Z] - z1[f - v.Z];
    st_c8(u, U.rcap, r, f, x);
  }
}

__global__ void __launch_bounds__(ROW_THREADS) clf_u_kernel(DevView v) {
  TraceScope trace_scope(v.trace, v.trace_id);
  clf_u_row(v, blockIdx.y, blockIdx.x * ROW_WARPS + (threadIdx.x >> 5), threadIdx.x & 31);
}

// ---------------------------------------------------------------------------------------------
// z3_post: per (row, class) evaluation e.  Sample the top latent and take fb(KL(q || N(0,I)))
// (DrVAE.py:341-345, VFAE.py:242-246).  grid (ceil(Fcap / ROW_WARPS), n_models)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void eval_decode(const DevView& v, int m, int e, int Fl, int& l, int& i, int& jj) {
  l = e / Fl;
  const int el = e - l * Fl;
  i = v.e_row.at(m)[el];
  jj = v.e_jj.at(m)[el];
}

template <int J>
__device__ __forceinline__ void z3_post_row(const DevView& v, const int m, const int e, const int lane) {
  const int* cnt = v.counts.at(m);
  const int F = cnt[CNT_F], Fl = cnt[CNT_FL];
  if (e >= pad128(F)) return;
  if (e >= F) {
    zero_c8_row(v.Z3b, m, e, lane);
    return;
  }
  int l, i, jj;
  eval_decode(v, m, e, Fl, l, i, jj);
  const float* q3 = v.Q3.at(m) + (long long)e * 2 * v.Z3s;
  const float* ez = v.eps_z3.at(m) + (((long long)l * v.Ncap + i) * v.Y + jj) * v.Z3;
  bf16* z3b = v.Z3b.at(m);
  const int cls = v.e_cls_full.at(m)[e];
  float a_mu[J], a_lv[J], a_ez[J];
#pragma unroll
  for (int k = 0; k < J; ++k) {  // every load of the row before the first store
    const int f = lane + 32 * k;
    const bool in = f < v.Z3;
    a_mu[k] = in ? q3[f] : 0.f;
    a_lv[k] = in ? q3[v.Z3s + f] : 0.f;
    a_ez[k] = in ? ez[f] : 0.f;
  }
  float kl = 0.f;
#pragma unroll
  for (int k = 0; k < J; ++k) {
    const int f = lane + 32 * k;
    if (f >= v.Z3c) continue;
    float z = (f == v.Z3 || f == v.Z3 + 1 + cls) ? 1.f : 0.f;  // ones column, one-hot class column
    if (f < v.Z3) {
      z = a_mu[k] + expf(0.5f * a_lv[k]) * a_ez[k];
      kl += kl_prior_term(a_mu[k], a_lv[k]);
    }
    st_c8(z3b, v.Z3b.rcap, e, f, z);
  }
  for (int f = 32 * J + lane; f < v.Z3c; f += 32)  // constant columns past the register slots (see sample_q1_row)
    st_c8(z3b, v.Z3b.rcap, e, f, (f == v.Z3 || f == v.Z3 + 1 + cls) ? 1.f : 0.f);
  kl = warp_sum(kl);
  if (lane == 0) v.kfp_row.at(m)[e] = fmaxf(kl, v.dyn->s.kl_min);
}

template <int J>
__global__ void __launch_bounds__(ROW_THREADS, ROW_LB_EVAL) z3_post_kernel(DevView v) {
  TraceScope trace_scope(v.trace, v.trace_id);
  z3_post_row<J>(v, blockIdx.y, blockIdx.x * ROW_WARPS + (threadIdx.x >> 5), threadIdx.x & 31);
}

// weight of evaluation e in the batch KLD: 1 for the true class of a labeled row, q(y=j) otherwise
__device__ __forceinline__ float eval_weight(const DevView& v, int m, int l, int i, int jj, int N) {
  if (v.lab.at(m)[i]) return 1.f;
  return v.QY.at(m)[((long long)l * N + i) * v.Y + jj];
}

// ---------------------------------------------------------------------------------------------
// pz1_post: fb(KL(q(z1|x1) || p(z1|z_top,y))) per evaluation, its gradients towards the
// decoder_z1 heads (dY9) and towards q1 (dQ1e).  DrVAE.py:352-355, VFAE.py:253-256.
// ---------------------------------------------------------------------------------------------
template <int J>
__device__ __forceinline__ void pz1_post_row(const DevView& v, const int m, const int e, const int lane) {
  const int* cnt = v.counts.at(m);
  const int N = cnt[CNT_N], F = cnt[CNT_F], Fl = cnt[CNT_FL];
  if (e >= pad128(F)) return;
  if (e >= F) {
    if (v.need_grad) zero_c8_row(v.dY9, m, e, lane);
    return;
  }
  int l, i, jj;
  eval_decode(v, m, e, Fl, l, i, jj);
  const float* q1 = v.Q.at(m) + (long long)i * 2 * v.Zs;
  const float* pz = v.PZ1.at(m) + (long long)e * 2 * v.Zs;
  float a_m1[J], a_l1[J], a_mp[J], a_lp[J];
#pragma unroll
  for (int k = 0; k < J; ++k) {  // every load of the row before the reduction
    const int f = lane + 32 * k;
    const bool in = f < v.Z;
    a_m1[k] = in ? q1[f] : 0.f;
    a_l1[k] = in ? q1[v.Zs + f] : 0.f;
    a_mp[k] = in ? pz[f] : 0.f;
    a_lp[k] = in ? pz[v.Zs + f] : 0.f;
  }
  const float w = eval_weight(v, m, l, i, jj, N);
  const float k3 = v.kfp_row.at(m)[e];
  float kl = 0.f;
#pragma unroll
  for (int k = 0; k < J; ++k)
    if (lane + 32 * k < v.Z) kl += kl_term(a_m1[k], a_l1[k], a_mp[k], a_lp[k]);
  kl = warp_sum(kl);
  const bool act = kl > v.dyn->s.kl_min;
  const float ke = k3 + fmaxf(kl, v.dyn->s.kl_min);
  __syncwarp();
  if (lane == 0) {
    v.kfp_row.at(m)[e] = ke;
    v.kfpw_row.at(m)[e] = w * ke;
  }
  if (!v.need_grad) return;
  const float cw = act ? v.coefs.at(m)[COEF_KLD] * w : 0.f;
  bf16* dy = v.dY9.at(m);
  float* dq = v.dQ1e.at(m) + (long long)e * 2 * v.Zs;
#pragma unroll
  for (int k = 0; k < J; ++k) {
    const int f = lane + 32 * k;
    if (f >= v.Z) continue;
    const float mu1 = a_m1[k], lv1 = a_l1[k], mup = a_mp[k], lvp = a_lp[k];
    const float d = mu1 - mup, ie = expf(-lvp), ev = expf(lv1);
    st_c8(dy, v.dY9.rcap, e, f, -cw * d * ie);
    st_c8(dy, v.dY9.rcap, e, v.Zs + f, cw * 0.5f * (1.f - (d * d + ev) * ie));
    dq[f] = cw * d * ie;
    dq[v.Zs + f] = cw * 0.5f * (ev * ie - 1.f);
  }
  zero_c8_gaps(v.dY9, dy, e, v.Z, v.Zs, lane);
}

template <int J>
__global__ void __launch_bounds__(ROW_THREADS, ROW_LB_EVAL) pz1_post_kernel(DevView v) {
  TraceScope trace_scope(v.trace, v.trace_id);
  pz1_post_row<J>(v, blockIdx.y, blockIdx.x * ROW_WARPS + (threadIdx.x >> 5), threadIdx.x & 31);
}

// ---------------------------------------------------------------------------------------------
// z3_back: d loss / d (mu3 | lv3) per evaluation = reparameterisation path (dZ3 from the
// decoder_z1 input gradient) + the direct prior-KL gradient.
// ---------------------------------------------------------------------------------------------
template <int J>
__device__ __forceinline__ void z3_back_row(const DevView& v, const int m, const int e, const int lane) {
  const int* cnt = v.counts.at(m);
  const int N = cnt[CNT_N], F = cnt[CNT_F], Fl = cnt[CNT_FL];
  if (e >= pad128(F)) return;
  if (e >= F) {
    zero_c8_row(v.dY7, m, e, lane);
    return;
  }
  int l, i, jj;
  eval_decode(v, m, e, Fl, l, i, jj);
  const float* q3 = v.Q3.at(m) + (long long)e * 2 * v.Z3s;
  const float* ez = v.eps_z3.at(m) + (((long long)l * v.Ncap + i) * v.Y + jj) * v.Z3;
  const float* dz = v.dZ3.at(m) + (long long)e * v.Z3;
  float a_mu[J], a_lv[J], a_ez[J], a_g[J];
#pragma unroll
  for (int k = 0; k < J; ++k) {  // every load of the row before the reduction
    const int f = lane + 32 * k;
    const bool in = f < v.Z3;
    a_mu[k] = in ? q3[f] : 0.f;
    a_lv[k] = in ? q3[v.Z3s + f] : 0.f;
    a_ez[k] = in ? ez[f] : 0.f;
    a_g[k] = in ? dz[f] : 0.f;
  }
  const float w = eval_weight(v, m, l, i, jj, N);
  float kl = 0.f;
#pragma unroll
  for (int k = 0; k < J; ++k)
    if (lane + 32 * k < v.Z3) kl += kl_prior_term(a_mu[k], a_lv[k]);
  kl = warp_sum(kl);
  const float cw = kl > v.dyn->s.kl_min ? v.coefs.at(m)[COEF_KLD] * w : 0.f;
  bf16* dy = v.dY7.at(m);
#pragma unroll
  for (int k = 0; k < J; ++k) {
    const int f = lane + 32 * k;
    if (f >= v.Z3) continue;
    const float mu = a_mu[k], lv = a_lv[k];
    const float g = a_g[k];
    st_c8(dy, v.dY7.rcap, e, f, g + cw * mu);
    st_c8(dy, v.dY7.rcap, e, v.Z3s + f, g * 0.5f * expf(0.5f * lv) * a_ez[k] + cw * 0.5f * (expf(lv) - 1.f));
  }
  zero_c8_gaps(v.dY7, dy, e, v.Z3, v.Z3s, lane);
}

template <int J>
__global__ void __launch_bounds__(ROW_THREADS, ROW_LB_EVAL) z3_back_kernel(DevView v) {
  TraceScope trace_scope(v.trace, v.trace_id);
  z3_back_row<J>(v, blockIdx.y, blockIdx.x * ROW_WARPS + (threadIdx.x >> 5), threadIdx.x & 31);
}

// ---------------------------------------------------------------------------------------------
// clf_back: d loss / d logits of q(y|.), pushed back to z1 (DZ1) and z2f (DZ2F).
//   labeled row   : -yloss_rate/(L max(1,Nlab)) * d log q_y
//   unlabeled row : 1/(L N) * d [ sum_j q_j k_j + sum_j q_j (log q_j - log prior_j) ]
// grid (ceil(LNcap / ROW_WARPS), n_models), one warp per stacked row r = l*N + i
// ---------------------------------------------------------------------------------------------
// d loss / d logits of row r = l * N + i (every lane computes the same values; lane 0 stores them for the weight gradient)
__device__ __forceinline__ void clf_dlogit_row(const DevView& v, const int m, const int r, const int l, const int i, const int Fl, const int lane,
                                               float (&dl)[MAXY]) {
  const float* cf = v.coefs.at(m);
  const float* qy = v.QY.at(m) + (long long)r * v.Y;
  const bool lb = v.lab.at(m)[i] != 0;
  const int yi = v.ycls.at(m)[i];
  float q[MAXY], g[MAXY];
  float dot = 0.f;
#pragma unroll
  for (int j = 0; j < MAXY; ++j) {
    q[j] = 0.f;
    g[j] = 0.f;
    if (j < v.Y) {
      q[j] = qy[j];
      // (the clamp's upper bound 1 - 1e-10 rounds to 1.0f, which no probability exceeds: only the lower bound can
      // cut a class's gradient, as in the reference's float32 clamp backward)
      const bool clamped = !(q[j] > 1e-10f);
      if (lb) {
        g[j] = (j == yi) ? -cf[COEF_YL] / q[j] : 0.f;
      } else {
        const float ke = v.has_fprop ? v.kfp_row.at(m)[l * Fl + v.ebase.at(m)[i] + j] : 0.f;
        g[j] = cf[COEF_KLD] * (ke + logf(q[j]) - v.member(m).log_prior[j] + 1.f);
      }
      if (clamped) g[j] = 0.f;
      dot += q[j] * g[j];
    }
  }
#pragma unroll
  for (int j = 0; j < MAXY; ++j) {
    dl[j] = (j < v.Y) ? q[j] * (g[j] - dot) : 0.f;
    if (j < v.Y && lane == 0) v.dlogit.at(m)[(long long)r * v.Y + j] = dl[j];
  }
}

__device__ __forceinline__ void clf_back_row(const DevView& v, const int m, const int r, const int lane) {
  const int* cnt = v.counts.at(m);
  const int N = cnt[CNT_N], LN = cnt[CNT_LN], Fl = cnt[CNT_FL];
  if (r >= LN) return;
  const int l = r / N, i = r - l * N;
  float dl[MAXY];
  clf_dlogit_row(v, m, r, l, i, Fl, lane, dl);
  const float* Wc = v.clf_w.at(m);
  const bool two = v.clf_in > v.Z;
  // (unrolled over the feature slots: the weight loads of all slots are in flight together)
#pragma unroll
  for (int k = 0; k < MAXJ; ++k) {
    const int f = lane + 32 * k;
    if (f >= v.Z) break;
    float a = 0.f, b = 0.f;
#pragma unroll
    for (int j = 0; j < MAXY; ++j) {
      if (j < v.Y) {
        a = fmaf(dl[j], Wc[j * v.clf_ld + f], a);
        if (two) b = fmaf(dl[j], Wc[j * v.clf_ld + v.Z + f], b);
      }
    }
    v.DZ1.at(m)[(long long)r * v.Z + f] = a - b;
    if (two) v.DZ2F.at(m)[(long long)r * v.Z + f] = b;
  }
}

__global__ void __launch_bounds__(ROW_THREADS) clf_back_kernel(DevView v) {
  TraceScope trace_scope(v.trace, v.trace_id);
  clf_back_row(v, blockIdx.y, blockIdx.x * ROW_WARPS + (threadIdx.x >> 5), threadIdx.x & 31);
}

// The same with hidden layers: d loss / d logits, then dPre of the last hidden layer, (dl . W_p) * ELU'(H) as bf16
// chunk8, with zero rows [LN, pad128(LN)) (the weight-gradient GEMMs contract over them).  The block's dX / dW GEMMs
// and clf_du take it from there.  grid (ceil(pad128(LNcap) / ROW_WARPS), n_models)
__device__ __forceinline__ void clf_back_h_row(const DevView& v, const int m, const int r, const int lane) {
  const int* cnt = v.counts.at(m);
  const int N = cnt[CNT_N], LN = cnt[CNT_LN], Fl = cnt[CNT_FL];
  const ClfView& cv = *v.clf;
  if (r >= LN) {
    if (r < pad128(LN)) zero_c8_row(cv.D, m, r, lane);
    return;
  }
  const int l = r / N, i = r - l * N;
  float dl[MAXY];
  clf_dlogit_row(v, m, r, l, i, Fl, lane, dl);
  const float* Wc = v.clf_w.at(m);
  const uint4* hp = reinterpret_cast<const uint4*>(cv.H.at(m)) + r;
  uint4* dp = reinterpret_cast<uint4*>(cv.D.at(m)) + r;
  for (int c = lane; c < (cv.D.fcap >> 3); c += 32) {
    float h[8], d[8];
    unpack_bf16x8(hp[(long long)c * cv.H.rcap], h);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int f = 8 * c + e;
      float g = 0.f;
      if (f < cv.pin) {
#pragma unroll
        for (int j = 0; j < MAXY; ++j)
          if (j < v.Y) g = fmaf(dl[j], Wc[j * v.clf_ld + f], g);
      }
      d[e] = f < cv.pin ? g * elu1_grad_from_out(h[e]) : 0.f;
    }
    dp[(long long)c * cv.D.rcap] = pack_bf16x8(d);
  }
}

__global__ void __launch_bounds__(ROW_THREADS) clf_back_h_kernel(DevView v) {
  TraceScope trace_scope(v.trace, v.trace_id);
  clf_back_h_row(v, blockIdx.y, blockIdx.x * ROW_WARPS + (threadIdx.x >> 5), threadIdx.x & 31);
}

// clf_du (DrVAE, hidden layers): d loss / d u = [dz1 part | dz2f part] from the first layer's dX GEMM ->
// DZ1 = dU[:Z] - dU[Z:], DZ2F = dU[Z:] (what clf_back_row writes without hidden layers).  One warp per stacked row.
__device__ __forceinline__ void clf_du_row(const DevView& v, const int m, const int r, const int lane) {
  if (r >= v.counts.at(m)[CNT_LN]) return;
  const float* du = v.clf->dU.at(m) + (long long)r * v.clf_in;
  for (int f = lane; f < v.Z; f += 32) {
    const float a = du[f], b = du[v.Z + f];
    v.DZ1.at(m)[(long long)r * v.Z + f] = a - b;
    v.DZ2F.at(m)[(long long)r * v.Z + f] = b;
  }
}

__global__ void __launch_bounds__(ROW_THREADS) clf_du_kernel(DevView v) {
  TraceScope trace_scope(v.trace, v.trace_id);
  clf_du_row(v, blockIdx.y, blockIdx.x * ROW_WARPS + (threadIdx.x >> 5), threadIdx.x & 31);
}

// ---------------------------------------------------------------------------------------------
// T_back: gradient rows of the p(z2|z1) heads (dYT = [d p_mu | d p_lv]), the KL(q2||p) gradient
// towards q2 (dQ2) and the residual / classifier contributions to d z1 (DZ1).
// ---------------------------------------------------------------------------------------------
template <int J>
__device__ __forceinline__ void T_back_row(const DevView& v, const int m, const int i, const int lane) {
  const int* cnt = v.counts.at(m);
  const int N = cnt[CNT_N], Np = cnt[CNT_NP], LN = cnt[CNT_LN], LNp = cnt[CNT_LNP];
  if (i >= N) {
    const int j = i - N;
    if (j < PAD_WARPS)
      for (int jj = j; jj < PAD_ROWS; jj += PAD_WARPS)
        if (LN + jj < pad128(LN)) zero_c8_row(v.dYT, m, LN + jj, lane);
    return;
  }
  const int p = v.pair_of.at(m)[i];
  const float* q2 = p >= 0 ? v.Q.at(m) + (long long)(N + p) * 2 * v.Zs : nullptr;
  const float ckl = v.coefs.at(m)[COEF_KLZ2];
  bf16* dy = v.dYT.at(m);
  float a_mu[J], a_lv[J], q2m[J], q2l[J];
#pragma unroll
  for (int k = 0; k < J; ++k) {
    const int f = lane + 32 * k;
    a_mu[k] = a_lv[k] = 0.f;
    q2m[k] = (q2 && f < v.Z) ? q2[f] : 0.f;
    q2l[k] = (q2 && f < v.Z) ? q2[v.Zs + f] : 0.f;
  }
  for (int l = 0; l < v.L; ++l) {
    const int r = l * N + i;
    const float* pt = v.PT.at(m) + (long long)r * 2 * v.Zs;
    const float* ef = v.eps_z2f.at(m) + ((long long)l * v.Ncap + i) * v.Z;
    const float* dzd = p >= 0 ? v.dZdec.at(m) + (long long)(LN + LNp + l * Np + p) * v.Z : nullptr;
    const bool act = q2 && v.klz2_row.at(m)[r] > v.dyn->s.kl_min;
    float* dz1 = v.DZ1.at(m) + (long long)r * v.Z;
    const float* dz2f_c = v.has_clf ? v.DZ2F.at(m) + (long long)r * v.Z : nullptr;
    float b_pmu[J], b_plv[J], b_g[J], b_c[J], b_ef[J], b_dz1[J];
#pragma unroll
    for (int k = 0; k < J; ++k) {  // every load of this sample before the first store
      const int f = lane + 32 * k;
      const bool in = f < v.Z;
      b_pmu[k] = in ? pt[f] : 0.f;
      b_plv[k] = in ? pt[v.Zs + f] : 0.f;
      b_g[k] = (in && dzd) ? dzd[f] : 0.f;
      b_c[k] = (in && dz2f_c) ? dz2f_c[f] : 0.f;
      b_ef[k] = in ? ef[f] : 0.f;
      b_dz1[k] = (in && v.has_clf) ? dz1[f] : 0.f;
    }
#pragma unroll
    for (int k = 0; k < J; ++k) {
      const int f = lane + 32 * k;
      if (f < v.Z) {
        const float pmu = b_pmu[k], plv = b_plv[k];
        float g = b_g[k] + b_c[k];
        float dpmu = g;
        float dplv = g * 0.5f * expf(0.5f * plv) * b_ef[k];
        if (act) {
          const float mu2 = q2m[k], lv2 = q2l[k];
          const float d = mu2 - pmu, ie = expf(-plv), ev = expf(lv2);
          dpmu += -ckl * d * ie;
          dplv += ckl * 0.5f * (1.f - (d * d + ev) * ie);
          a_mu[k] += ckl * d * ie;
          a_lv[k] += ckl * 0.5f * (ev * ie - 1.f);
        }
        dz1[f] = b_dz1[k] + dpmu;  // residual path mu = z1 + ...
        st_c8(dy, v.dYT.rcap, r, f, dpmu);
        st_c8(dy, v.dYT.rcap, r, v.Zs + f, dplv);
      }
    }
    zero_c8_gaps(v.dYT, dy, r, v.Z, v.Zs, lane);
  }
  if (p >= 0) {
    float* dq2 = v.dQ2.at(m) + (long long)p * 2 * v.Zs;
#pragma unroll
    for (int k = 0; k < J; ++k) {
      const int f = lane + 32 * k;
      if (f < v.Z) {
        dq2[f] = a_mu[k];
        dq2[v.Zs + f] = a_lv[k];
      }
    }
  }
}

template <int J>
__global__ void __launch_bounds__(ROW_THREADS, ROW_LB_TBACK) T_back_kernel(DevView v) {
  TraceScope trace_scope(v.trace, v.trace_id);
  T_back_row<J>(v, blockIdx.y, blockIdx.x * ROW_WARPS + (threadIdx.x >> 5), threadIdx.x & 31);
}

// ---------------------------------------------------------------------------------------------
// q_back: gradient rows of the encoder heads, dY2 = [d mu | d lv] for q(z1|x1) rows and for
// q(z2|x2) rows.  Collects every path into z1 / z2 samples and the direct KL gradients.
// ---------------------------------------------------------------------------------------------
template <int J>
__device__ __forceinline__ void q_back_row(const DevView& v, const int m, const int i, const int lane) {
  const int* cnt = v.counts.at(m);
  const int N = cnt[CNT_N], Np = cnt[CNT_NP], LN = cnt[CNT_LN], R0 = cnt[CNT_R0], Fl = cnt[CNT_FL];
  if (i >= N) {
    const int j = i - N;
    if (j < PAD_WARPS)
      for (int jj = j; jj < PAD_ROWS; jj += PAD_WARPS)
        if (R0 + jj < pad128(R0)) zero_c8_row(v.dY2, m, R0 + jj, lane);
    return;
  }
  const float* q = v.Q.at(m) + (long long)i * 2 * v.Zs;
  const int p = v.pair_of.at(m)[i];
  const int eb = v.has_fprop ? v.ebase.at(m)[i] : 0;
  const int ecnt = v.has_fprop ? (v.lab.at(m)[i] ? 1 : v.Y) : 0;
  const bool have_dz1 = v.has_clf || v.has_T;
  bf16* dy = v.dY2.at(m);
  const float cN = v.coefs.at(m)[COEF_INV_N];
  const bool pv = v.kind == KIND_PVAE;
  const float klq1 = pv ? v.klq_row.at(m)[i] : 0.f;
  const float klq2 = (pv && p >= 0) ? v.klq_row.at(m)[N + p] : 0.f;
  // Feature f = lane + 32 k.  Per MC sample all gradient rows of this minibatch row are requested together (one
  // memory round trip per sample and per class evaluation instead of one per feature slot, sample and evaluation);
  // the sums run in the same order as the reference accumulation: sample-major, evaluations in class order.
  float mu[J], lv[J], hs[J], amu[J], alv[J];
#pragma unroll
  for (int k = 0; k < J; ++k) {
    const int f = lane + 32 * k;
    mu[k] = f < v.Z ? q[f] : 0.f;
    lv[k] = f < v.Z ? q[v.Zs + f] : 0.f;
    amu[k] = alv[k] = 0.f;
  }
#pragma unroll
  for (int k = 0; k < J; ++k) hs[k] = 0.5f * expf(0.5f * lv[k]);
  for (int l = 0; l < v.L; ++l) {
    const long long r = (long long)l * N + i;
    const float* gd = v.dZdec.at(m) + r * v.Z;
    const float* g1 = v.DZ1.at(m) + r * v.Z;
    const float* gT = v.dZ1T.at(m) + r * v.Z;
    const float* e1 = v.eps_z1.at(m) + ((long long)l * v.Ncap + i) * v.Z;
    const float* g2p = v.dZdec.at(m) + ((long long)LN + (long long)l * Np + p) * v.Z;
    const float* e2 = v.eps_z2.at(m) + ((long long)l * v.Ncap + i) * v.Z;
    float g[J], a_e1[J], a_g2[J], a_e2[J];
#pragma unroll
    for (int k = 0; k < J; ++k) {
      const int f = lane + 32 * k;
      const bool in = f < v.Z;
      float x = in ? gd[f] : 0.f;
      const float y1 = (in && have_dz1) ? g1[f] : 0.f;
      const float yT = (in && v.has_T) ? gT[f] : 0.f;
      a_e1[k] = in ? e1[f] : 0.f;
      a_g2[k] = (in && p >= 0) ? g2p[f] : 0.f;
      a_e2[k] = (in && p >= 0) ? e2[f] : 0.f;
      if (have_dz1) x += y1;
      if (v.has_T) x += yT;
      g[k] = x;
    }
    for (int jj = 0; jj < ecnt; ++jj) {
      const long long e = (long long)l * Fl + eb + jj;
      const float* ze = v.dZ1e.at(m) + e * v.Z;
      const float* qe = v.dQ1e.at(m) + e * 2 * v.Zs;
      float a_ze[J], a_qm[J], a_ql[J];
#pragma unroll
      for (int k = 0; k < J; ++k) {
        const int f = lane + 32 * k;
        const bool in = f < v.Z;
        a_ze[k] = in ? ze[f] : 0.f;
        a_qm[k] = in ? qe[f] : 0.f;
        a_ql[k] = in ? qe[v.Zs + f] : 0.f;
      }
#pragma unroll
      for (int k = 0; k < J; ++k) {
        g[k] += a_ze[k];
        amu[k] += a_qm[k];
        alv[k] += a_ql[k];
      }
    }
#pragma unroll
    for (int k = 0; k < J; ++k) {
      amu[k] += g[k];
      alv[k] += g[k] * hs[k] * a_e1[k];
      if (p >= 0) {
        amu[k] += a_g2[k];
        alv[k] += a_g2[k] * hs[k] * a_e2[k];
      }
    }
  }
  const float* q2 = v.Q.at(m) + (long long)(N + (p >= 0 ? p : 0)) * 2 * v.Zs;
  const float* dq2 = v.dQ2.at(m) + (long long)(p >= 0 ? p : 0) * 2 * v.Zs;
#pragma unroll
  for (int k = 0; k < J; ++k) {
    const int f = lane + 32 * k;
    if (f >= v.Z) continue;
    if (pv && klq1 > v.dyn->s.kl_min) {
      amu[k] += cN * mu[k];
      alv[k] += cN * 0.5f * (expf(lv[k]) - 1.f);
    }
    st_c8(dy, v.dY2.rcap, i, f, amu[k]);
    st_c8(dy, v.dY2.rcap, i, v.Zs + f, alv[k]);
    if (p >= 0) {
      float bmu = v.has_T ? dq2[f] : 0.f;
      float blv = v.has_T ? dq2[v.Zs + f] : 0.f;
      if (pv && klq2 > v.dyn->s.kl_min) {
        bmu += cN * q2[f];
        blv += cN * 0.5f * (expf(q2[v.Zs + f]) - 1.f);
      }
      st_c8(dy, v.dY2.rcap, N + p, f, bmu);
      st_c8(dy, v.dY2.rcap, N + p, v.Zs + f, blv);
    }
  }
  zero_c8_gaps(v.dY2, dy, i, v.Z, v.Zs, lane);
  if (p >= 0) zero_c8_gaps(v.dY2, dy, N + p, v.Z, v.Zs, lane);
}

template <int J>
__global__ void __launch_bounds__(ROW_THREADS, ROW_LB_QBACK) q_back_kernel(DevView v) {
  TraceScope trace_scope(v.trace, v.trace_id);
  q_back_row<J>(v, blockIdx.y, blockIdx.x * ROW_WARPS + (threadIdx.x >> 5), threadIdx.x & 31);
}

// ---------------------------------------------------------------------------------------------
// classifier weight gradient: dWc[j][t] = sum_r dlogit[r][j] * u[r][t], u = [z1, z2f - z1, 1] (with hidden layers
// u = [H_last, 1], the bf16 activation the logits were computed from)
// two stages (row-split partials, then a fixed-order reduction) -> deterministic
// ---------------------------------------------------------------------------------------------
// (m, split): one row split of one model; thread t0 of nthreads cooperating threads
// with hidden layers: u = [H_last, 1]
__device__ __forceinline__ void clf_grad_partial_h_block(const DevView& v, const int m, const int split, const int t0, const int nthreads) {
  const ClfView& cv = *v.clf;
  const int LN = v.counts.at(m)[CNT_LN], splits = v.clf_splits, Y = v.Y;
  const float* dlogit = v.dlogit.at(m);
  float* part = v.clf_part.at(m);
  const int width = cv.pin + 1;
  for (int t = t0; t < width; t += nthreads) {
    float acc[MAXY];
#pragma unroll
    for (int j = 0; j < MAXY; ++j) acc[j] = 0.f;
    for (int r = split; r < LN; r += splits) {
      const float u = t < cv.pin ? __bfloat162float(cv.H.at(m)[c8_index(r, t, cv.H.rcap)]) : 1.f;
      const float* dl = dlogit + (long long)r * Y;
#pragma unroll
      for (int j = 0; j < MAXY; ++j)
        if (j < Y) acc[j] = fmaf(dl[j], u, acc[j]);
    }
#pragma unroll
    for (int j = 0; j < MAXY; ++j)
      if (j < Y) part[((long long)split * Y + j) * width + t] = acc[j];
  }
}

__device__ __forceinline__ void clf_grad_partial_block(const DevView& v, const int m, const int split, const int t0, const int nthreads) {
  const int LN = v.counts.at(m)[CNT_LN];
  const int width = v.clf_in + 1;
  for (int t = t0; t < width; t += nthreads) {
    float acc[MAXY];
#pragma unroll
    for (int j = 0; j < MAXY; ++j) acc[j] = 0.f;
    for (int r = split; r < LN; r += v.clf_splits) {
      float u;
      if (t < v.Z)
        u = v.Z1f.at(m)[(long long)r * v.Z + t];
      else if (t < v.clf_in)
        u = v.Z2Ff.at(m)[(long long)r * v.Z + t - v.Z] - v.Z1f.at(m)[(long long)r * v.Z + t - v.Z];
      else
        u = 1.f;
      const float* dl = v.dlogit.at(m) + (long long)r * v.Y;
#pragma unroll
      for (int j = 0; j < MAXY; ++j)
        if (j < v.Y) acc[j] = fmaf(dl[j], u, acc[j]);
    }
#pragma unroll
    for (int j = 0; j < MAXY; ++j)
      if (j < v.Y) v.clf_part.at(m)[((long long)split * v.Y + j) * width + t] = acc[j];
  }
}

__global__ void __launch_bounds__(256) clf_grad_partial_kernel(DevView v) {
  TraceScope trace_scope(v.trace, v.trace_id);
  clf_grad_partial_block(v, blockIdx.y, blockIdx.x, threadIdx.x, 256);
}

__global__ void __launch_bounds__(256) clf_grad_partial_h_kernel(DevView v) {
  TraceScope trace_scope(v.trace, v.trace_id);
  clf_grad_partial_h_block(v, blockIdx.y, blockIdx.x, threadIdx.x, 256);
}

// grid (ceil(Y * (clf_in + 1) / 8), n_models), block 256: one warp per gradient element, lanes over the row splits
// (lane l sums splits l, l + 32, ... in order, then a fixed shuffle tree -> deterministic)
__device__ __forceinline__ void clf_grad_reduce_elem(const DevView& v, const int m, const int k, const int lane) {
  const int pin = v.clf ? v.clf->pin : v.clf_in;  // input width of linear_p
  const int width = pin + 1;
  if (k >= v.Y * width) return;
  const int j = k / width, t = k - j * width;
  float s = 0.f;
  for (int sp = lane; sp < v.clf_splits; sp += 32) s += v.clf_part.at(m)[((long long)sp * v.Y + j) * width + t];
  s = warp_sum(s);
  if (lane != 0) return;
  const int idx = (t < pin) ? v.clf_w_off + j * v.clf_ld + t : v.clf_b_off + j;
  if (!v.dyn->s.fused_adam) {
    v.grads.at(m)[idx] = s;
  } else {
    // the classifier runs on the fp32 parameters directly: Adam here, no shadow to refresh
    float* P = v.params.at(m);
    float* M1 = v.adam_m.at(m);
    float* V2 = v.adam_v.at(m);
    float pv = P[idx], m1 = M1[idx], v1 = V2[idx];
    adam_update(s, pv, m1, v1, v.member(m).adam);
    M1[idx] = m1;
    V2[idx] = v1;
    P[idx] = pv;
  }
}

__global__ void __launch_bounds__(256) clf_grad_reduce_kernel(DevView v) {
  TraceScope trace_scope(v.trace, v.trace_id);
  clf_grad_reduce_elem(v, blockIdx.y, blockIdx.x * 8 + (threadIdx.x >> 5), threadIdx.x & 31);
}


// ---------------------------------------------------------------------------------------------
// inference (DrVAE.forward, DrVAE.py:253-311): deterministic mu path, no sampling
// ---------------------------------------------------------------------------------------------
struct InferView {
  float *z1_mu, *z1_lv, *z2_mu, *z2_lv, *proba;
  int* pred;
};

__global__ void infer_counts_kernel(DevView v, int rows_dec) {
  const int m = blockIdx.x;
  if (threadIdx.x == 0) {
    int* cnt = v.counts.at(m);
    cnt[CNT_N] = v.N;
    cnt[CNT_NP] = 0;
    cnt[CNT_NLAB] = 0;
    cnt[CNT_R0] = v.N;
    cnt[CNT_LN] = v.N;
    cnt[CNT_LNP] = 0;
    cnt[CNT_RD] = rows_dec;
    cnt[CNT_FL] = 0;
    cnt[CNT_F] = 0;
  }
  for (int i = threadIdx.x; i < v.N; i += blockDim.x) {
    v.lab.at(m)[i] = 0;
    v.ycls.at(m)[i] = 0;
  }
}

__device__ __forceinline__ void infer_emit_proba(const DevView& v, const InferView& o, int m, int r, int lane) {
  if (lane == 0) {
    const float* q = v.QY.at(m) + (long long)r * v.Y;
    int best = 0;
    for (int j = 0; j < v.Y; ++j) {
      if (o.proba) o.proba[((long long)m * v.N + r) * v.Y + j] = q[j];
      if (q[j] > q[best]) best = j;
    }
    if (o.pred) o.pred[(long long)m * v.N + r] = best;
  }
}

// z1 = mu(q(z1|x1)); stage it for the p(z2|z1) and decoder GEMMs.  One warp per row.
__global__ void __launch_bounds__(ROW_THREADS) infer_z1_kernel(DevView v, InferView o, int rows_dec) {
  const int m = blockIdx.y, lane = threadIdx.x & 31;
  const int r = blockIdx.x * ROW_WARPS + (threadIdx.x >> 5);
  const int N = v.N;
  if (r >= N) {
    const int j = r - N;
    if (j < PAD_WARPS)
      for (int jj = j; jj < PAD_ROWS; jj += PAD_WARPS)
        if (rows_dec + jj < pad128(rows_dec)) zero_c8_row(v.Zdec, m, rows_dec + jj, lane);
    return;
  }
  const float* q = v.Q.at(m) + (long long)r * 2 * v.Zs;
  bf16* zdec = v.Zdec.at(m);
  for (int f = lane; f < v.Zc; f += 32) {
    float z = 0.f;
    if (f < v.Z) {
      z = q[f];
      v.Z1f.at(m)[(long long)r * v.Z + f] = z;
      if (o.z1_mu) o.z1_mu[((long long)m * N + r) * v.Z + f] = z;
      if (o.z1_lv) o.z1_lv[((long long)m * N + r) * v.Z + f] = q[v.Zs + f];
    }
    st_c8(zdec, v.Zdec.rcap, r, f, z);
  }
  if (v.has_clf && !v.has_T && !v.clf) {
    __syncwarp();
    classifier_row(v, m, r, r, lane);
    __syncwarp();
    infer_emit_proba(v, o, m, r, lane);
  }
}

// z2 = mu(p(z2|z1)) = z1 + z1 W^T + b; classifier on [z1, z2 - z1].
__global__ void __launch_bounds__(ROW_THREADS) infer_z2_kernel(DevView v, InferView o) {
  const int m = blockIdx.y, lane = threadIdx.x & 31;
  const int r = blockIdx.x * ROW_WARPS + (threadIdx.x >> 5);
  const int N = v.N;
  if (r >= N) return;
  const float* pt = v.PT.at(m) + (long long)r * 2 * v.Zs;
  const float* z1 = v.Z1f.at(m) + (long long)r * v.Z;
  bf16* zdec = v.Zdec.at(m);
  for (int f = lane; f < v.Zc; f += 32) {
    float z = 0.f;
    if (f < v.Z) {
      z = z1[f] + pt[f];
      v.Z2Ff.at(m)[(long long)r * v.Z + f] = z;
      if (o.z2_mu) o.z2_mu[((long long)m * N + r) * v.Z + f] = z;
      if (o.z2_lv) o.z2_lv[((long long)m * N + r) * v.Z + f] = pt[v.Zs + f];
    }
    st_c8(zdec, v.Zdec.rcap, N + r, f, z);
    if (v.clf && f < v.Z) {  // u = [z1 | z2 - z1] for the classifier's hidden layers (clf_h_infer_kernel)
      st_c8(v.clf->U.at(m), v.clf->U.rcap, r, f, z1[f]);
      st_c8(v.clf->U.at(m), v.clf->U.rcap, r, v.Z + f, z - z1[f]);
    }
  }
  if (v.has_clf && !v.clf) {
    __syncwarp();
    classifier_row(v, m, r, r, lane);
    __syncwarp();
    infer_emit_proba(v, o, m, r, lane);
  }
}

// classifier with hidden layers: logits from the last hidden activation (the block's GEMMs ran over u)
__global__ void __launch_bounds__(ROW_THREADS) clf_h_infer_kernel(DevView v, InferView o) {
  const int m = blockIdx.y, lane = threadIdx.x & 31;
  const int r = blockIdx.x * ROW_WARPS + (threadIdx.x >> 5);
  if (r >= v.N) return;
  classifier_row_h(v, m, r, r, lane);
  __syncwarp();
  infer_emit_proba(v, o, m, r, lane);
}

// ---------------------------------------------------------------------------------------------
// loss: fixed-order reduction of the per-row terms into the reference's loss dictionary
// (DrVAE.py:610-626, PVAE.py:452-465, VFAE.py:438-458).  out: RECL KLD PERT YL MMD ELBO CMPL.
// With global normalisers (data parallel) the outputs are this shard's additive share.
// ---------------------------------------------------------------------------------------------
// sum over 256 cooperating threads (t = 0 .. 255) in a fixed tree order; `sync` is the barrier of exactly those threads
// (__syncthreads in the stand-alone kernel, a named barrier inside the persistent step kernel)
struct SyncBlock {
  __device__ __forceinline__ void operator()() const { __syncthreads(); }
};
template <class Sync>
__device__ __forceinline__ float block_sum_256(float x, float* sm, const int t, const Sync& sync) {
  sm[t] = x;
  sync();
  for (int o = 128; o > 0; o >>= 1) {
    if (t < o) sm[t] += sm[t + o];
    sync();
  }
  const float r = sm[0];
  sync();
  return r;
}

// grid (loss_slices, n_models): slice s reduces rows s, s + slices, ... of every per-row term in a fixed order
// (m, slice) of `nslices`: 256 cooperating threads, t = 0 .. 255
template <class Sync>
__device__ __forceinline__ void loss_partial_block(const DevView& v, const int m, const int slice, const int nslices, const int t, float* sm,
                                                   const Sync& sync) {
  const int stride = 256 * nslices, first = slice * 256 + t;
  const int* cnt = v.counts.at(m);
  const int LN = cnt[CNT_LN], LNp = cnt[CNT_LNP], Rd = cnt[CNT_RD], F = cnt[CNT_F], R0 = cnt[CNT_R0];
  float a_recl = 0.f, a_pert = 0.f;
  for (int r = first; r < Rd; r += stride) {
    float s = 0.f;
    for (int k = 0; k < v.dec_tiles; ++k) s += v.dec_part.at(m)[(long long)k * v.Rdcap + r];
    if (r < LN + LNp)
      a_recl += s;
    else
      a_pert += s;
  }
  float a_klz2 = 0.f, a_yl = 0.f, a_ycat = 0.f, a_kfp = 0.f, a_klq = 0.f;
  for (int r = first; r < LN; r += stride) {
    if (v.has_T) a_klz2 += v.klz2_row.at(m)[r];
    if (v.has_clf) {
      a_yl += v.yl_row.at(m)[r];
      a_ycat += v.ycat_row.at(m)[r];
    }
  }
  if (v.has_fprop)
    for (int e = first; e < F; e += stride) a_kfp += v.kfpw_row.at(m)[e];
  if (v.kind == KIND_PVAE)
    for (int r = first; r < R0; r += stride) a_klq += v.klq_row.at(m)[r];
  a_recl = block_sum_256(a_recl, sm, t, sync);
  a_pert = block_sum_256(a_pert, sm, t, sync);
  a_klz2 = block_sum_256(a_klz2, sm, t, sync);
  a_yl = block_sum_256(a_yl, sm, t, sync);
  a_ycat = block_sum_256(a_ycat, sm, t, sync);
  a_kfp = block_sum_256(a_kfp, sm, t, sync);
  a_klq = block_sum_256(a_klq, sm, t, sync);
  if (t == 0) {
    float* o = v.loss_part.at(m) + slice * 8;
    o[0] = a_recl, o[1] = a_pert, o[2] = a_klz2, o[3] = a_yl, o[4] = a_ycat, o[5] = a_kfp, o[6] = a_klq, o[7] = 0.f;
  }
}

__global__ void __launch_bounds__(256) loss_partial_kernel(DevView v) {
  TraceScope trace_scope(v.trace, v.trace_id);
  __shared__ float sm[256];
  loss_partial_block(v, blockIdx.y, blockIdx.x, gridDim.x, threadIdx.x, sm, SyncBlock());
}

// grid n_models, one warp: fixed-order sum of the slices, then the reference's normalisation
// one thread per model
__device__ __forceinline__ void loss_final_model(const DevView& v, const int m) {
  float a[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int s = 0; s < v.loss_slices; ++s)
    for (int k = 0; k < 7; ++k) a[k] += v.loss_part.at(m)[s * 8 + k];
  const float* cf = v.coefs.at(m);
  const float RECL = cf[COEF_RECL] * a[0];
  const float PERT = cf[COEF_PERT_PLAIN] * a[1];
  const float KLD = cf[COEF_KLZ2] * a[2] + cf[COEF_KLD] * (a[5] + a[4]) + cf[COEF_INV_N] * a[6];
  const float YL = cf[COEF_YL_PLAIN] * a[3];
  const MemberScalars& ms = v.member(m);
  const float ELBO = RECL + v.dyn->s.beta_pert * ms.pertloss_rate * PERT - KLD;
  const float CMPL = -ELBO - ms.yloss_rate * YL;
  float* o = v.losses.at(m);
  o[0] = RECL;
  o[1] = KLD;
  o[2] = PERT;
  o[3] = YL;
  o[4] = 0.f;
  o[5] = ELBO;
  o[6] = CMPL;
  o[7] = 0.f;
}

__global__ void __launch_bounds__(32) loss_final_kernel(DevView v) {
  TraceScope trace_scope(v.trace, v.trace_id);
  if (threadIdx.x == 0) loss_final_model(v, blockIdx.x);
}

}  // namespace drvae
