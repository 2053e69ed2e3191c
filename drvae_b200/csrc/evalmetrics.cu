// Metrics of the evaluation path (SURVEY.md §8(f) rank 1) on the device, for one model or all E members of an ensemble.
//
// Reference: DeepGenerativeModelMixin.eval_x_reconstruction / eval_y_prediction, src/DGMMixin.py:128-190 — numpy
// float64 RMSE, sklearn.metrics.r2_score(multioutput='variance_weighted'), a Python loop of scipy.stats.pearsonr over
// the rows, the mean per-row Gaussian log-likelihood (src/blocks.py:230-234), and sklearn's roc_auc_score /
// average_precision_score on the class probabilities.  It runs on the full train and validation sets every epoch
// (src/DrVAE.py:784-821); once the training step takes microseconds that loop dominates an epoch.
//
// Reconstruction: three small kernels, blockIdx.y (rows, columns) or blockIdx.x (final) = member, all arithmetic in
// fp64 like the reference, every reduction in a fixed order (deterministic):
//   eval_rows_kernel   one warp per selected row: sums of x, r, x^2, r^2, x r, (x - r)^2 and of the log-density terms
//                      -> Pearson r, squared error and log-likelihood of the row
//   eval_cols_kernel   one thread per feature: sum and sum of squares of x over the selected rows (the variance-weighted
//                      R^2 needs the total sum of squares around the per-feature means)
//   eval_final_kernel  one block per member: fixed-order sums of the row and column statistics -> {rmse, r2, pearr, ll}
//
// Ranking (AUROC, average precision) in the counting form, no sort: for every positive row i of a score column,
//   nlt_i = negatives with score < s_i, neq_i = negatives with score == s_i, tp_i = positives with score >= s_i,
//   fp_i = negatives with score >= s_i;
//   AUROC = sum_i (nlt_i + neq_i / 2) / (P Nn)   (the trapezoid under sklearn's ROC curve, tied scores one step)
//   AP    = sum_i tp_i / (tp_i + fp_i) / P       (sklearn's step-wise average precision)
// The counts are integers (exact); the precision terms are summed in a fixed order.  Three kernels:
//   rank_prep_kernel   one block per member: labeled-row count, correct predictions, the nan conditions, and per score
//                      column a stable partition of the labeled rows' scores (positives from the front, negatives from
//                      the back of a D-float slot)
//   rank_count_kernel  (positive chunk, column, member): 1024 positives per block against every labeled row, streamed
//                      through shared memory in tiles -> per-block partial sums
//   rank_final_kernel  one thread per member: partials in chunk order -> {acc, auroc, aupr}
#include <cuda_runtime.h>
#include <math.h>

#include "drvae_b200.h"
#include "errors.h"

namespace {

constexpr int kCols = 11;           // drvae_eval_members output columns
constexpr int kRankThreads = 256;   // rank_count_kernel block
constexpr int kRankPerThread = 4;   // positives per thread
constexpr int kRankChunk = kRankThreads * kRankPerThread;
constexpr int kRankTile = 2048;     // scores per shared-memory tile
constexpr int kPrepThreads = 1024;  // rank_prep_kernel block

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// rowstats[m][i] = {pearson r, sum (x - r)^2, log-likelihood, selected ? 1 : 0}; member m = blockIdx.y, its rows start
// at m * N.  A row is selected when mask (if any) and mask2 (if any) are non-zero.
__global__ void __launch_bounds__(256) eval_rows_kernel(const float* __restrict__ x, const float* __restrict__ r, const float* __restrict__ sg,
                                                        const int* __restrict__ mask, const int* __restrict__ mask2, int N, int X,
                                                        double* __restrict__ rowstats) {
  const int i = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (i >= N) return;
  const long long row = (long long)blockIdx.y * N + i;
  double* o = rowstats + 4 * row;
  if ((mask && mask[row] == 0) || (mask2 && mask2[row] == 0)) {
    if (lane < 4) o[lane] = 0.0;
    return;
  }
  const float* xr = x + row * X;
  const float* rr = r + row * X;
  const float* sr = sg ? sg + row * X : nullptr;
  double sx = 0, sy = 0, sxx = 0, syy = 0, sxy = 0, se = 0, ll = 0;
  const double LOG2PI = 1.8378770664093454836;
  for (int f = lane; f < X; f += 32) {
    const double a = xr[f], b = rr[f];
    sx += a;
    sy += b;
    sxx += a * a;
    syy += b * b;
    sxy += a * b;
    const double d = a - b;
    se += d * d;
    if (sr) {
      const double s = sr[f];
      ll += -0.5 * (LOG2PI + log(s * s) + d * d / (s * s));
    }
  }
  sx = warp_sum_d(sx);
  sy = warp_sum_d(sy);
  sxx = warp_sum_d(sxx);
  syy = warp_sum_d(syy);
  sxy = warp_sum_d(sxy);
  se = warp_sum_d(se);
  ll = warp_sum_d(ll);
  if (lane == 0) {
    const double n = X;
    const double cov = sxy - sx * sy / n, vx = sxx - sx * sx / n, vy = syy - sy * sy / n;
    o[0] = cov / sqrt(vx * vy);  // zero variance -> nan, like scipy.stats.pearsonr
    o[1] = se;
    o[2] = sr ? ll : nan("");
    o[3] = 1.0;
  }
}

// colstats[m][f] = {sum_i x[m][i][f], sum_i x[m][i][f]^2} over the selected rows of member m = blockIdx.y
__global__ void __launch_bounds__(128) eval_cols_kernel(const float* __restrict__ x, const int* __restrict__ mask, const int* __restrict__ mask2,
                                                        int N, int X, double* __restrict__ colstats) {
  const int f = blockIdx.x * 128 + threadIdx.x;
  if (f >= X) return;
  const long long m0 = (long long)blockIdx.y * N;
  double s = 0, ss = 0;
  for (int i = 0; i < N; ++i) {
    if ((mask && mask[m0 + i] == 0) || (mask2 && mask2[m0 + i] == 0)) continue;
    const double a = x[(m0 + i) * X + f];
    s += a;
    ss += a * a;
  }
  double* c = colstats + 2 * ((long long)blockIdx.y * X + f);
  c[0] = s;
  c[1] = ss;
}

__device__ double block_sum_d(double v, double* sm) {
  const int t = threadIdx.x;
  sm[t] = v;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (t < o) sm[t] += sm[t + o];
    __syncthreads();
  }
  const double r = sm[0];
  __syncthreads();
  return r;
}

// member m = blockIdx.x: out[m * out_stride + 0..3] = {rmse, r2, pearr, ll}
__global__ void __launch_bounds__(256) eval_final_kernel(const double* __restrict__ rowstats, const double* __restrict__ colstats, int N, int X,
                                                         double* __restrict__ out, int out_stride) {
  __shared__ double sm[256];
  const int t = threadIdx.x;
  rowstats += 4LL * N * blockIdx.x;
  colstats += 2LL * X * blockIdx.x;
  out += (long long)out_stride * blockIdx.x;
  double pr = 0, se = 0, ll = 0, cnt = 0;
  for (int i = t; i < N; i += 256) {
    const double* o = rowstats + 4 * (long long)i;
    if (o[3] != 0.0) {
      pr += o[0];
      se += o[1];
      ll += o[2];
      cnt += 1.0;
    }
  }
  pr = block_sum_d(pr, sm);
  se = block_sum_d(se, sm);
  ll = block_sum_d(ll, sm);
  cnt = block_sum_d(cnt, sm);
  double tot = 0;
  for (int f = t; f < X; f += 256) tot += colstats[2 * f + 1] - colstats[2 * f] * colstats[2 * f] / cnt;
  tot = block_sum_d(tot, sm);
  if (t == 0) {
    out[0] = cnt > 0 ? sqrt(se / (cnt * X)) : nan("");
    out[1] = (cnt > 0 && tot > 0) ? 1.0 - se / tot : nan("");
    out[2] = cnt > 0 ? pr / cnt : nan("");
    out[3] = cnt > 0 ? ll / cnt : nan("");
  }
}

__global__ void eval_fill_nan_kernel(double* __restrict__ out, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = nan("");
}

// Per member (blockIdx.x): mstats[m] = {labeled rows, correct predictions, nan flag (a label outside [0, Y) or a
// non-finite score in a scored column)}, ccount[m][c] = {P, Nn}, and for every score column c the labeled rows'
// scores in part[m][c][0..D): positives at [0, P) in row order, negatives at [D - Nn, D) in reverse row order.  Binary
// (Y == 2): one column, the score is proba[:, 1]; otherwise C = Y columns, one-vs-rest.
__global__ void __launch_bounds__(kPrepThreads) rank_prep_kernel(const int* __restrict__ valid, const int* __restrict__ has_y,
                                                                 const int* __restrict__ y, const int* __restrict__ pred,
                                                                 const float* __restrict__ proba, int D, int Y, int C,
                                                                 float* __restrict__ part, int* __restrict__ mstats, int* __restrict__ ccount) {
  __shared__ int wpos[kPrepThreads / 32], wneg[kPrepThreads / 32];
  const int m = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const unsigned lt_mask = (1u << lane) - 1u;
  const long long r0 = (long long)m * D;
  int n = 0, correct = 0, bad = 0;
  for (int c = 0; c < C; ++c) {
    const int cls = C == 1 ? 1 : c;
    float* dst = part + ((long long)m * C + c) * D;
    int np = 0, nn = 0;
    for (int i0 = 0; i0 < D; i0 += kPrepThreads) {
      const int i = i0 + t;
      const bool lab = i < D && valid[r0 + i] != 0 && has_y[r0 + i] != 0;
      const int label = lab ? y[r0 + i] : -1;
      const float s = lab ? proba[(r0 + i) * Y + cls] : 0.f;
      if (c == 0) {
        bool nonfinite = false;
        if (lab) {
          if (C == 1) {
            nonfinite = !isfinite(s);
          } else {
            for (int k = 0; k < Y; ++k) nonfinite |= !isfinite(proba[(r0 + i) * Y + k]);
          }
        }
        n += __syncthreads_count(lab);
        correct += __syncthreads_count(lab && pred[r0 + i] == label);
        bad |= __syncthreads_or(lab && (label < 0 || label >= Y || nonfinite));
      }
      const bool pos = lab && label == cls, neg = lab && label != cls;
      const unsigned bp = __ballot_sync(0xffffffffu, pos), bn = __ballot_sync(0xffffffffu, neg);
      if (lane == 0) {
        wpos[warp] = __popc(bp);
        wneg[warp] = __popc(bn);
      }
      __syncthreads();
      int op = np, on = nn;
      for (int w = 0; w < kPrepThreads / 32; ++w) {
        if (w == warp) {
          op += __popc(bp & lt_mask);
          on += __popc(bn & lt_mask);
        }
        const int a = wpos[w], b = wneg[w];
        if (w < warp) {
          op += a;
          on += b;
        }
        np += a;
        nn += b;
      }
      if (pos) dst[op] = s;
      if (neg) dst[D - 1 - on] = s;
      __syncthreads();
    }
    if (t == 0) {
      ccount[2 * (m * C + c)] = np;
      ccount[2 * (m * C + c) + 1] = nn;
    }
  }
  if (t == 0) {
    mstats[3 * m] = n;
    mstats[3 * m + 1] = correct;
    mstats[3 * m + 2] = bad;
  }
}

// Counts of src[0..cnt) below (and at or below, LE) each of the thread's scores, streamed in tiles.  Tile slots past
// cnt hold +inf, which no finite score exceeds or equals.
template <bool LE>
__device__ __forceinline__ void rank_count_tiles(const float* __restrict__ src, int cnt, const float (&si)[kRankPerThread],
                                                 int (&lt)[kRankPerThread], int (&le)[kRankPerThread], float* tile) {
  for (int j0 = 0; j0 < cnt; j0 += kRankTile) {
    __syncthreads();
    for (int j = threadIdx.x; j < kRankTile; j += kRankThreads) tile[j] = j0 + j < cnt ? src[j0 + j] : INFINITY;
    __syncthreads();
    const float4* t4 = reinterpret_cast<const float4*>(tile);
    const int n4 = min(kRankTile, cnt - j0 + 3) / 4;
#pragma unroll 4
    for (int j = 0; j < n4; ++j) {
      const float4 v = t4[j];
#pragma unroll
      for (int k = 0; k < kRankPerThread; ++k) {
        lt[k] += (v.x < si[k]) + (v.y < si[k]) + (v.z < si[k]) + (v.w < si[k]);
        if (LE) le[k] += (v.x <= si[k]) + (v.y <= si[k]) + (v.z <= si[k]) + (v.w <= si[k]);
      }
    }
  }
}

// Block (chunk, c, m): the positives [chunk * kRankChunk, +kRankChunk) of column c of member m against all labeled
// rows.  -> ap_part / auc_part[(m * C + c) * chunks + chunk] = {sum tp/(tp+fp), sum (2 nlt + neq)} over its positives.
__global__ void __launch_bounds__(kRankThreads) rank_count_kernel(const float* __restrict__ part, const int* __restrict__ mstats,
                                                                  const int* __restrict__ ccount, int D, int C, int chunks,
                                                                  double* __restrict__ ap_part, long long* __restrict__ auc_part) {
  __shared__ __align__(16) float tile[kRankTile];
  __shared__ double sap[kRankThreads];
  __shared__ long long sauc[kRankThreads];
  const int chunk = blockIdx.x, c = blockIdx.y, m = blockIdx.z, t = threadIdx.x;
  const int mc = m * C + c;
  const int P = ccount[2 * mc], Nn = ccount[2 * mc + 1];
  const int p0 = chunk * kRankChunk;
  if (mstats[3 * m + 2] != 0 || p0 >= P) return;  // nan result, or no positive in this chunk
  const float* src = part + (long long)mc * D;
  float si[kRankPerThread];
  int nlt[kRankPerThread], nle[kRankPerThread], plt[kRankPerThread], unused[kRankPerThread];
#pragma unroll
  for (int k = 0; k < kRankPerThread; ++k) {
    const int p = p0 + k * kRankThreads + t;
    si[k] = p < P ? src[p] : 0.f;
    nlt[k] = nle[k] = plt[k] = 0;
  }
  rank_count_tiles<true>(src + (D - Nn), Nn, si, nlt, nle, tile);
  rank_count_tiles<false>(src, P, si, plt, unused, tile);
  double ap = 0;
  long long auc = 0;
#pragma unroll
  for (int k = 0; k < kRankPerThread; ++k) {
    if (p0 + k * kRankThreads + t < P) {
      const int tp = P - plt[k], fp = Nn - nlt[k];
      ap += (double)tp / (double)(tp + fp);
      auc += 2LL * nlt[k] + (nle[k] - nlt[k]);
    }
  }
  sap[t] = ap;
  sauc[t] = auc;
  __syncthreads();
  for (int o = kRankThreads / 2; o > 0; o >>= 1) {
    if (t < o) {
      sap[t] += sap[t + o];
      sauc[t] += sauc[t + o];
    }
    __syncthreads();
  }
  if (t == 0) {
    ap_part[(long long)mc * chunks + chunk] = sap[0];
    auc_part[(long long)mc * chunks + chunk] = sauc[0];
  }
}

// out[m][0..2] = {accuracy, macro AUROC, macro AP} (the degenerate cases of training.eval_y_prediction: no labeled row
// -> nan; a column without positives or without negatives -> AUROC nan; a column without positives -> AP 0).
__global__ void rank_final_kernel(const int* __restrict__ mstats, const int* __restrict__ ccount, const double* __restrict__ ap_part,
                                  const long long* __restrict__ auc_part, int E, int C, int chunks, double* __restrict__ out) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= E) return;
  const int n = mstats[3 * m], correct = mstats[3 * m + 1], bad = mstats[3 * m + 2];
  double* o = out + (long long)kCols * m;
  o[0] = n > 0 ? (double)correct / (double)n : nan("");
  if (n == 0 || bad) {
    o[1] = o[2] = nan("");
    return;
  }
  double auroc = 0, aupr = 0;
  for (int c = 0; c < C; ++c) {
    const int mc = m * C + c;
    const int P = ccount[2 * mc], Nn = ccount[2 * mc + 1];
    double ap = 0;
    long long auc = 0;
    for (int k = 0; k < (P + kRankChunk - 1) / kRankChunk; ++k) {
      ap += ap_part[(long long)mc * chunks + k];
      auc += auc_part[(long long)mc * chunks + k];
    }
    auroc += (P > 0 && Nn > 0) ? (double)auc / (2.0 * (double)P * (double)Nn) : nan("");
    aupr += P > 0 ? ap / P : 0.0;
  }
  o[1] = auroc / C;
  o[2] = aupr / C;
}

// Reconstruction metrics of E members (rows selected by mask and mask2) -> out[m * out_stride + 0..3].
void launch_reconstruction(const float* x, const float* r, const float* sg, const int* mask, const int* mask2, int E, int N, int X,
                           double* out, int out_stride, double* ws, cudaStream_t st) {
  double* rowstats = ws;
  double* colstats = rowstats + 4LL * E * N;
  eval_rows_kernel<<<dim3((N + 7) / 8, E), 256, 0, st>>>(x, r, sg, mask, mask2, N, X, rowstats);
  eval_cols_kernel<<<dim3((X + 127) / 128, E), 128, 0, st>>>(x, mask, mask2, N, X, colstats);
  eval_final_kernel<<<E, 256, 0, st>>>(rowstats, colstats, N, X, out, out_stride);
}

long long recon_ws_bytes(int E, int D, int X) { return (long long)sizeof(double) * E * (4LL * D + 2LL * X); }

int rank_columns(int Y) { return Y == 2 ? 1 : Y; }
int rank_chunks(int D) { return (D + kRankChunk - 1) / kRankChunk; }

}  // namespace

extern "C" long long drvae_eval_workspace_bytes(int N, int X) {
  if (N < 1 || X < 1) return -1;
  return recon_ws_bytes(1, N, X);
}

extern "C" int drvae_eval_x_reconstruction(const float* x, const float* x_rec, const float* x_sigma, const int* mask, int N, int X,
                                           double* out, void* workspace, void* stream) {
  if (!x || !x_rec || !out || !workspace) return drvae::set_error("drvae_eval_x_reconstruction: null argument");
  if (N < 1 || X < 1) return drvae::set_error("drvae_eval_x_reconstruction: empty input");
  cudaStream_t st = (cudaStream_t)stream;
  launch_reconstruction(x, x_rec, x_sigma, mask, nullptr, 1, N, X, out, 4, reinterpret_cast<double*>(workspace), st);
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) return drvae::set_cuda_error("drvae_eval_x_reconstruction", err);
  return 0;
}

extern "C" long long drvae_eval_members_workspace_bytes(int E, int D, int X, int Y) {
  if (E < 1 || D < 1 || X < 1) return -1;
  long long b = recon_ws_bytes(E, D, X);
  if (Y >= 2) {
    const long long C = rank_columns(Y), parts = (long long)E * C * rank_chunks(D);
    b += parts * (sizeof(double) + sizeof(long long)) + sizeof(float) * E * C * (long long)D + sizeof(int) * (3LL * E + 2LL * E * C);
  }
  return b;
}

extern "C" int drvae_eval_members(const drvae_eval_members_in_t* in, int E, int D, int X, int Y, double* out, void* workspace,
                                  void* stream) {
  if (!in) return drvae::set_error("drvae_eval_members: in is NULL");
  if (!in->valid) return drvae::set_error("drvae_eval_members: valid is NULL");
  if (!out) return drvae::set_error("drvae_eval_members: out is NULL");
  if (!workspace) return drvae::set_error("drvae_eval_members: workspace is NULL");
  if (E < 1 || E > 65535) return drvae::set_error("drvae_eval_members: E must be in [1, 65535]");
  if (D < 1) return drvae::set_error("drvae_eval_members: D must be >= 1");
  if (X < 1) return drvae::set_error("drvae_eval_members: X must be >= 1");
  const bool g1 = in->x1 || in->px1_mu || in->px1_sg;
  if (g1 && !(in->x1 && in->px1_mu)) return drvae::set_error("drvae_eval_members: x1 group needs x1 and px1_mu");
  const bool g2 = in->x2 || in->px2_mu || in->px2_sg || in->has_x2;
  if (g2 && !(in->x2 && in->px2_mu && in->has_x2)) return drvae::set_error("drvae_eval_members: x2 group needs x2, px2_mu and has_x2");
  const bool gy = in->proba || in->pred || in->y || in->has_y;
  if (gy && !(in->proba && in->pred && in->y && in->has_y)) return drvae::set_error("drvae_eval_members: y group needs proba, pred, y and has_y");
  if (gy && Y < 2) return drvae::set_error("drvae_eval_members: Y must be >= 2 with the y group");
  cudaStream_t st = (cudaStream_t)stream;
  double* ws = reinterpret_cast<double*>(workspace);
  if (!(g1 && g2 && gy)) eval_fill_nan_kernel<<<(E * kCols + 255) / 256, 256, 0, st>>>(out, E * kCols);
  // the x1 and x2 passes share one reconstruction region (stream order)
  if (g1) launch_reconstruction(in->x1, in->px1_mu, in->px1_sg, in->valid, nullptr, E, D, X, out + 3, kCols, ws, st);
  if (g2) launch_reconstruction(in->x2, in->px2_mu, in->px2_sg, in->valid, in->has_x2, E, D, X, out + 7, kCols, ws, st);
  if (gy) {
    const int C = rank_columns(Y), chunks = rank_chunks(D);
    double* ap_part = reinterpret_cast<double*>(reinterpret_cast<char*>(workspace) + recon_ws_bytes(E, D, X));
    long long* auc_part = reinterpret_cast<long long*>(ap_part + (long long)E * C * chunks);
    float* part = reinterpret_cast<float*>(auc_part + (long long)E * C * chunks);
    int* mstats = reinterpret_cast<int*>(part + (long long)E * C * D);
    int* ccount = mstats + 3LL * E;
    rank_prep_kernel<<<E, kPrepThreads, 0, st>>>(in->valid, in->has_y, in->y, in->pred, in->proba, D, Y, C, part, mstats, ccount);
    rank_count_kernel<<<dim3(chunks, C, E), kRankThreads, 0, st>>>(part, mstats, ccount, D, C, chunks, ap_part, auc_part);
    rank_final_kernel<<<(E + 127) / 128, 128, 0, st>>>(mstats, ccount, ap_part, auc_part, E, C, chunks, out);
  }
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) return drvae::set_cuda_error("drvae_eval_members", err);
  return 0;
}
