// Optimizer-side kernels: the stand-alone Adam pass over the flat parameter vector (torch.optim.Adam
// semantics, SURVEY.md Appendix A.6 / reference DGMMixin.py:31-40, :123; drvae_train_step fuses the
// same update into the weight-gradient epilogues instead) that also refreshes the derived
// kernel-facing copies (bf16 chunk8 weight shadows, fp32 bias / class-bias vectors), the
// weight-norm row kernels, and the Philox ε generator.
#pragma once

#include "plan.h"

namespace drvae {

__device__ __forceinline__ int seg_find(const Seg* segs, int nseg, int idx) {
  int lo = 0, hi = nseg - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (segs[mid].off <= idx)
      lo = mid;
    else
      hi = mid - 1;
  }
  return lo;
}

// Write the kernel-facing copy of parameter element `idx` (value `pv`) of model m.
__device__ __forceinline__ void write_derived(const Seg& s, int idx, float pv, bf16* shadow, float* derived) {
  if (s.kind == SEG_W) {
    if (s.wn_g_off >= 0) return;  // weight-normalised layers: shadow = g v / ||v||, written row-wise
    const int local = idx - s.off;
    const int n = local / s.ld, k = local - n * s.ld;
    if (k >= s.cols) return;  // row padding
    const int srow = (n / s.ilv_block) * s.ilv_stride + s.which * s.ilv_block + (n % s.ilv_block);
    if (k < s.kmain)
      shadow[s.sh_off + c8_index(srow, k, s.sh_rcap)] = __float2bfloat16_rn(pv);
    else
      derived[s.clsb_off + (long long)(k - s.kmain) * s.clsb_ld + srow] = pv;
  } else if (s.kind == SEG_B) {
    const int n = idx - s.off;
    const int srow = (n / s.ilv_block) * s.ilv_stride + s.which * s.ilv_block + (n % s.ilv_block);
    derived[s.bias_off + srow] = pv + s.bias_const;
  }
}

struct AdamArgs {
  MBuf<float> params, grads, m, v;
  MBuf<bf16> shadow;
  MBuf<float> derived;
  const Seg* segs;
  int nseg;
  int P;  // parameters per model
  const AdamHyper* h;  // device memory (StepDyn or the member table)
  int h_ms;            // bytes between the Adam scalars of consecutive models (0: shared)
  int update;  // 0: only refresh the derived copies from the current parameters
  // parameters [skip_lo, skip_hi) are left untouched when the batch (global counts if given) has no pair rows
  int skip_lo, skip_hi;
  const StepDyn* dyn;
  const int* counts;
  int counts_stride;
};

// grid (ceil(P / 1024), n_models), block 256, 4 elements per thread
__global__ void __launch_bounds__(256) adam_kernel(AdamArgs a) {
  const int mdl = blockIdx.y;
  float* p = a.params.at(mdl);
  const float* g = a.grads.p ? a.grads.at(mdl) : nullptr;
  float* mm = a.m.p ? a.m.at(mdl) : nullptr;
  float* vv = a.v.p ? a.v.at(mdl) : nullptr;
  bf16* sh = a.shadow.at(mdl);
  float* dv = a.derived.at(mdl);
  const int base = blockIdx.x * 1024 + threadIdx.x;
  AdamHyper hyper{};
  if (a.update) hyper = adam_of(a.h, a.h_ms, mdl);
  bool skip_range = false;
  if (a.update && a.skip_hi > a.skip_lo) {
    const int np = a.dyn->s.gN > 0 ? a.dyn->s.gNp : a.counts[(long long)mdl * a.counts_stride + CNT_NP];
    skip_range = np == 0;
  }
  int si = -1;
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int idx = base + u * 256;
    if (idx >= a.P) break;
    float pv = p[idx];
    if (a.update && !(skip_range && idx >= a.skip_lo && idx < a.skip_hi)) {
      float m1 = mm[idx], v1 = vv[idx];
      adam_update(g[idx], pv, m1, v1, hyper);
      mm[idx] = m1;
      vv[idx] = v1;
      p[idx] = pv;
    }
    if (si < 0 || idx < a.segs[si].off || (si + 1 < a.nseg && idx >= a.segs[si + 1].off)) si = seg_find(a.segs, a.nseg, idx);
    // tensors start on 16-byte boundaries: an index in the padding after a segment belongs to no tensor
    if (idx - a.segs[si].off < a.segs[si].rows * a.segs[si].ld) write_derived(a.segs[si], idx, pv, sh, dv);
  }
}

// ---------------------------------------------------------------------------------------------
// weight norm (layers.WeightNormLinear): one warp per output row of every normalised layer
// grid (ceil(rows / 8), n_models), block 256
// ---------------------------------------------------------------------------------------------
struct WnArgs {
  const WnRow* rows;
  int nrows;
  MBuf<float> params, grads;
  MBuf<bf16> shadow;
  MBuf<float> derived;
};

// effective rows -> bf16 shadow / class bias / classifier copy
__global__ void __launch_bounds__(256) wn_refresh_kernel(WnArgs a) {
  const int m = blockIdx.y, lane = threadIdx.x & 31;
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= a.nrows) return;
  const WnRow w = a.rows[r];
  const float* vrow = a.params.at(m) + w.w_off;
  float ss = 0.f;
  for (int k = lane; k < w.len; k += 32) ss += vrow[k] * vrow[k];
  ss = warp_sum(ss);
  const float scale = a.params.at(m)[w.g_idx] / sqrtf(ss);
  if (w.sh_off >= 0) {
    bf16* sh = a.shadow.at(m) + w.sh_off;
    for (int k = lane; k < w.kin; k += 32) sh[c8_index(w.srow, k, w.sh_rcap)] = __float2bfloat16_rn(scale * vrow[k]);
    float* cb = a.derived.at(m) + w.aux_off;
    for (int k = w.kin + lane; k < w.len; k += 32) cb[(long long)(k - w.kin) * w.aux_ld + w.srow] = scale * vrow[k];
  } else {
    float* eff = a.derived.at(m) + w.aux_off;
    for (int k = lane; k < w.len; k += 32) eff[k] = scale * vrow[k];
  }
}

// in place: gradient wrt the effective row -> gradient wrt v (same slots) and g
//   dg = <dW, v> / ||v|| ;  dv = (g / ||v||) dW - (g <dW, v> / ||v||^3) v
__global__ void __launch_bounds__(256) wn_grad_kernel(WnArgs a) {
  const int m = blockIdx.y, lane = threadIdx.x & 31;
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= a.nrows) return;
  const WnRow w = a.rows[r];
  const float* vrow = a.params.at(m) + w.w_off;
  float* grow = a.grads.at(m) + w.w_off;
  float ss = 0.f, dot = 0.f;
  for (int k = lane; k < w.len; k += 32) {
    const float vk = vrow[k];
    ss += vk * vk;
    dot += grow[k] * vk;
  }
  ss = warp_sum(ss);
  dot = warp_sum(dot);
  const float inv = 1.f / sqrtf(ss);
  const float g = a.params.at(m)[w.g_idx];
  const float c1 = g * inv, c2 = g * dot * inv * inv * inv;
  for (int k = lane; k < w.len; k += 32) grow[k] = c1 * grow[k] - c2 * vrow[k];
  if (lane == 0) a.grads.at(m)[w.g_idx] = dot * inv;
}

// test knob (drvae_debug_side_delay): holds a stream for `cycles` clocks so that a missing cross-stream dependency
// shows up as a wrong result instead of passing by timing luck
__global__ void spin_kernel(long long cycles) {
  const long long t0 = clock64();
  while (clock64() - t0 < cycles) __nanosleep(64);
}

// writes the per-step scalars; the only kernel whose arguments differ between two steps of the same shape.  With a
// member table it also expands the table into this step's per-member scalars: lr / bc1 rounds like the host's float
// division of adam_scalars(), so a member gets exactly the update of a table-less plan run with its lr.
__global__ void set_dyn_kernel(StepDyn value, StepDyn* dst, MemberExpand mx) {
  if (threadIdx.x == 0) {
    if (value.counts_dev) {  // batch-global normalisers left in device memory by the caller's all-reduce
      value.s.gN = (int)value.counts_dev[0];
      value.s.gNp = (int)value.counts_dev[1];
      value.s.gNlab = (int)value.counts_dev[2];
    }
    *dst = value;
  }
  for (int k = threadIdx.x; k < mx.n; k += blockDim.x) {
    const drvae_member_hparams_t h = mx.table[k];
    MemberScalars s;
    s.noise_std = h.noise_std;
    s.pertloss_rate = h.pertloss_rate;
    s.kl_qz2pz2_rate = h.kl_qz2pz2_rate;
    s.yloss_rate = h.yloss_rate;
#pragma unroll
    for (int j = 0; j < 8; ++j) s.log_prior[j] = h.log_prior_y[j];
    s.adam = value.s.mem.adam;
    s.adam.lr_bc1 = __fdiv_rn(h.lr, value.bc1);
    s.adam.wd = h.weight_decay;
    mx.out[k] = s;
  }
}

// ε block generator.  Every normal is keyed by (seed, step, model, segment, MC sample, GLOBAL row,
// position in the row) and never by its address, so a minibatch sharded over ranks
// (row_offset = global index of the shard's first row) draws exactly the noise of the unsharded
// run.  One thread = 4 consecutive normals of one row.  grid (blocks, n_models, 6 segments)
struct EpsSegs {
  long long off[6];  // segment offsets inside the per-model ε block (drvae_eps_layout_t order)
  int outer[6];      // MC samples (1 for the input-noise segments)
  int inner[6];      // floats per row
};

__global__ void __launch_bounds__(256) philox_normal_kernel(MBuf<float> out, EpsSegs sg, int N, int Ncap, const StepDyn* dyn,
                                                            unsigned long long* trace, int trace_id) {
  TraceScope trace_scope(trace, trace_id);
  const long long row_offset = dyn->row_offset;
  const unsigned long long seed = dyn->noise_seed;
  const unsigned int step = dyn->noise_step;
  const int m = blockIdx.y, seg = blockIdx.z;
  int inner = 0, outer = 0;
  long long seg_off = 0;
#pragma unroll
  for (int i = 0; i < 6; ++i)  // static indexing: a dynamic index would copy the struct to local memory
    if (i == seg) inner = sg.inner[i], outer = sg.outer[i], seg_off = sg.off[i];
  const int quads = (inner + 3) >> 2;
  const unsigned total = (unsigned)outer * (unsigned)N * (unsigned)quads;  // < 2^31 (checked on the host)
  const unsigned t = blockIdx.x * 256u + threadIdx.x;
  if (inner <= 0 || t >= total) return;
  const unsigned lr = t / (unsigned)quads;
  const int q = (int)(t - lr * (unsigned)quads);
  const int l = (int)(lr / (unsigned)N), r = (int)(lr - (unsigned)l * (unsigned)N);
  const unsigned long long grow = (unsigned long long)(row_offset + r);
  float z[4];
  philox_normal4(seed, step, m, seg, l, grow, q, z);
  float* o = out.at(m) + seg_off + ((long long)l * Ncap + r) * inner + q * 4;
  if (!(inner & 1) && !(seg_off & 1)) {  // even rows: 8-byte aligned pairs
    if (q * 4 + 1 < inner) *reinterpret_cast<float2*>(o) = make_float2(z[0], z[1]);
    if (q * 4 + 3 < inner) *reinterpret_cast<float2*>(o + 2) = make_float2(z[2], z[3]);
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (q * 4 + j < inner) o[j] = z[j];
  }
}

}  // namespace drvae
