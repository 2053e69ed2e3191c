// fp32 inference path (DrVAE.forward / PVAE.forward / VFAE.forward, reference src/DrVAE.py:253-311, src/PVAE.py:206-246,
// src/VFAE.py:178-215): the deterministic mu-path evaluated in full fp32 straight from the master parameters.
//
// Why it exists.  north_star asks for thresholded y-predictions that match the reference EXACTLY.  The training step
// runs its GEMMs with bf16 operands (1e-3 budget on the loss terms), which moves class probabilities by ~1e-3 and
// flips argmax on rows whose margin is smaller than that — about one row in a few hundred at the README dims.  Inference
// is not the hot path (forward only, once per evaluation), so it is evaluated with fp32 operands and fp32 FMA
// accumulation: probabilities agree with the reference to ~1e-6 and the thresholded predictions are identical
// (tests/test_shapes_gpu.py counts the mismatches on 150 and 8192 rows).  The bf16 tensor-core inference path stays
// available (drvae_set_infer_precision) for callers that prefer speed.
#pragma once

#include "plan.h"

namespace drvae {

enum { ACT_NONE = 0, ACT_ELU = 1, ACT_SOFTPLUS_EPS = 2, ACT_SOFTPLUS = 3 };  // ACT_SOFTPLUS: softplus hidden layers

struct LinF32 {
  const float* X;   // [rows][ldx]
  long long x_ms;
  int ldx;
  const float* W;   // [nout][ldw] (reference layout, row stride ldw)
  const float* b;   // [nout]
  long long p_ms;   // floats between models in the parameter vector
  int ldw;
  float bconst;     // folded constant (logvar heads: -2)
  const float* resid;  // optional [rows][ldr] added to the output (p(z2|z1): mu = z + z W^T + b)
  long long r_ms;
  int ldr;
  float* out;       // [rows][ldo]
  long long o_ms;
  int ldo;
  int rows, nout, K;
  int act;
};

// out[r][n] = act(sum_k X[r][k] W[n][k] + b[n] + bconst (+ resid[r][n])): 64 x 64 output tile per CTA, K in slabs of 16,
// 256 threads x (4 x 4) outputs, fp32 FMA.  grid (ceil(nout / 64), ceil(rows / 64), models)
__global__ void __launch_bounds__(256) linear_f32_kernel(LinF32 a) {
  __shared__ float Xs[16][64 + 4];
  __shared__ float Ws[16][64 + 4];
  const int m = blockIdx.z;
  const float* X = a.X + m * a.x_ms;
  const float* W = a.W + m * a.p_ms;
  const float* B = a.b + m * a.p_ms;
  const int r0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  const int lr = threadIdx.x >> 2, lk = (threadIdx.x & 3) * 4;  // loader: row 0..63, k offset 0, 4, 8, 12
  for (int k0 = 0; k0 < a.K; k0 += 16) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = k0 + lk + j;
      Xs[lk + j][lr] = (r0 + lr < a.rows && k < a.K) ? X[(long long)(r0 + lr) * a.ldx + k] : 0.f;
      Ws[lk + j][lr] = (n0 + lr < a.nout && k < a.K) ? W[(long long)(n0 + lr) * a.ldw + k] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      float xv[4], wv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) xv[i] = Xs[k][ty * 4 + i], wv[i] = Ws[k][tx * 4 + i];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(xv[i], wv[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = r0 + ty * 4 + i;
    if (r >= a.rows) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= a.nout) continue;
      float y = acc[i][j] + B[n] + a.bconst;
      if (a.resid) y += a.resid[m * a.r_ms + (long long)r * a.ldr + n];
      if (a.act == ACT_ELU) y = y > 0.f ? y : expm1f(y);
      if (a.act == ACT_SOFTPLUS_EPS) y = (y > 20.f ? y : log1pf(expf(y))) + 1e-3f;
      if (a.act == ACT_SOFTPLUS) y = y > 20.f ? y : log1pf(expf(y));
      a.out[m * a.o_ms + (long long)r * a.ldo + n] = y;
    }
  }
}

// u = [z1, z2 - z1] of DrVAE in fp32, [N][ld] (the input of the classifier's hidden layers).  grid (ceil(N 2Z / 256), models)
__global__ void __launch_bounds__(256) clf_u_f32_kernel(const float* z1, const float* z2, long long z_ms, int Z, int N, float* u,
                                                        long long u_ms, int ld) {
  const int m = blockIdx.y;
  const long long k = (long long)blockIdx.x * 256 + threadIdx.x;
  if (k >= (long long)N * 2 * Z) return;
  const int r = (int)(k / (2 * Z)), f = (int)(k - (long long)r * 2 * Z);
  const float* a = z1 + m * z_ms + (long long)r * Z;
  const float* b = z2 + m * z_ms + (long long)r * Z;
  u[m * u_ms + (long long)r * ld + f] = f < Z ? a[f] : b[f - Z] - a[f - Z];
}

// classifier q(y | u), u = [z1, z2 - z1] (DrVAE) or z1 (VFAE), on fp32 latents; writes proba / pred.  One warp per row.
// With hidden layers z1 is the last hidden activation (Z = its width, z2 = null).
struct ClfF32 {
  const float* z1;  // [N][ldz]
  const float* z2;  // [N][ldz] or null
  long long z_ms;
  int ldz;
  const float* W;   // [Y][ldw]
  const float* b;
  long long p_ms;
  int ldw, Z, Y, N;
  float* proba;     // [models][N][Y] or null
  int* pred;        // [models][N] or null
};

__global__ void __launch_bounds__(256) clf_f32_kernel(ClfF32 a) {
  const int m = blockIdx.y, lane = threadIdx.x & 31;
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= a.N) return;
  const float* z1 = a.z1 + m * a.z_ms + (long long)r * a.ldz;
  const float* z2 = a.z2 ? a.z2 + m * a.z_ms + (long long)r * a.ldz : nullptr;
  const float* W = a.W + m * a.p_ms;
  const float* B = a.b + m * a.p_ms;
  float acc[MAXY];
#pragma unroll
  for (int j = 0; j < MAXY; ++j) acc[j] = 0.f;
  for (int f = lane; f < a.Z; f += 32) {
    const float u = z1[f], d = z2 ? z2[f] - u : 0.f;
#pragma unroll
    for (int j = 0; j < MAXY; ++j) {
      if (j < a.Y) {
        acc[j] = fmaf(W[j * a.ldw + f], u, acc[j]);
        if (z2) acc[j] = fmaf(W[j * a.ldw + a.Z + f], d, acc[j]);
      }
    }
  }
  float mx = -INFINITY;
#pragma unroll
  for (int j = 0; j < MAXY; ++j) {
    if (j < a.Y) {
      acc[j] = warp_sum(acc[j]) + B[j];
      mx = fmaxf(mx, acc[j]);
    }
  }
  float den = 0.f;
#pragma unroll
  for (int j = 0; j < MAXY; ++j) {
    if (j < a.Y) {
      acc[j] = expf(acc[j] - mx);
      den += acc[j];
    }
  }
  if (lane != 0) return;
  int best = 0;
  float bq = -1.f;
#pragma unroll
  for (int j = 0; j < MAXY; ++j) {
    if (j < a.Y) {
      const float q = fminf(fmaxf(acc[j] / den, 1e-10f), 1.f - 1e-10f);  // blocks.py:462
      if (a.proba) a.proba[((long long)m * a.N + r) * a.Y + j] = q;
      if (q > bq) bq = q, best = j;  // torch.max: first maximal index
    }
  }
  if (a.pred) a.pred[(long long)m * a.N + r] = best;
}

}  // namespace drvae
