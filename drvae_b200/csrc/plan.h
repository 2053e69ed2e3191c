// Plan: everything the step executor needs for one ensemble of identically shaped models —
// parameter layout (reference state_dict order), bf16 weight shadows, workspace buffers, and the
// device-visible view of them that the row kernels take by value.
#pragma once

#include <string>
#include <vector>

#include "common.cuh"
#include "drvae_b200.h"
#include "gemm.cuh"

namespace drvae {

enum { KIND_DRVAE = 0, KIND_PVAE = 1, KIND_VFAE = 2 };

template <class T>
struct MBuf {  // one buffer per ensemble member, `ms` elements apart
  T* p;
  long long ms;
  __host__ __device__ __forceinline__ T* at(int model) const { return p + (long long)model * ms; }
};

// chunk8 bf16 buffer (per model)
struct C8Buf {
  bf16* p;
  long long ms;
  int rcap;
  int fcap;  // feature capacity (multiple of 8)
  __host__ __device__ __forceinline__ bf16* at(int model) const { return p + (long long)model * ms; }
};

// ---------------------------------------------------------------------------------------------
// parameter tensors and their derived (kernel-facing) copies
// ---------------------------------------------------------------------------------------------
enum { SEG_PLAIN = 0, SEG_W = 1, SEG_B = 2, SEG_G = 3 };

struct Seg {
  int off;   // offset in the flat per-model parameter vector
  int rows;  // out features (or vector length)
  int cols;  // in features (1 for vectors)
  int ld;    // floats between rows: cols rounded up to 4 (16-byte aligned rows; the padding stays zero)
  int kind;
  // SEG_W: bf16 chunk8 shadow [Kc/8][sh_rcap][8]; columns >= kmain are one-hot class columns
  long long sh_off;
  int sh_rcap;
  int kmain;
  int which, ilv_block, ilv_stride;
  long long clsb_off;  // fp32 [Y][clsb_ld]
  int clsb_ld;
  // SEG_B: fp32 derived bias vector, constant folded in
  long long bias_off;
  float bias_const;
  int wn_g_off;  // >= 0: weight-normalised layer, offset of its `g` vector (shadow written by wn kernel)
};

struct ParamInfo {
  std::string name;
  int rows, cols;  // cols == 0: vector
  int off;
  int ld;  // floats between rows (cols rounded up to a multiple of 4); 1 for vectors
};

// One weight matrix as the GEMMs see it (possibly two stacked / interleaved reference tensors).
struct Shadow {
  long long off;       // in the bf16 shadow arena (per model)
  int rcap;            // = tiles_n * BN  (output-feature capacity)
  int kin;             // true input features that go through the GEMM
  int kaug;            // kin + 1 (ones column -> bias gradient) + one-hot class columns
  int kc;              // round_up(kaug, 16): K extent of the forward GEMM, M extent of the dW GEMM
  int nout_total;      // shadow rows in use
  int BN, tiles_n;     // forward N tiling
  int BNx, tiles_nx;   // tiling over input features (dX / dW output columns)
  long long bias_off;  // fp32 derived bias [rcap]
  long long clsb_off;  // fp32 derived class bias [Y][rcap] or -1
  int ntens;
  int w_off[2];   // flat offsets of the weight tensors
  int b_off[2];   // flat offsets of the bias tensors
  int rows_each[2];
  int ld;         // leading dimension of the weight tensors: kin + class columns, rounded up to 4 (16-byte rows)
  int ilv_block, ilv_stride;
  float bias_const[2];  // constant folded into the derived bias (logvar heads: -2)
  long long tab_off;    // offset of this weight's 3 x rcap gradient-epilogue tables (EpiParams::g_tab)
  int g_off[2];         // weight norm: flat offsets of the `g` vectors (-1: plain nn.Linear)
};

// One output row of a weight-normalised layer (layers.WeightNormLinear, reference layers.py:25-41):
// effective weight row = g[n] / ||v[n, :]|| * v[n, :].  The kernels never see v: the bf16 shadow (and
// the class-bias / classifier copies) hold the effective row, refreshed by wn_refresh_kernel; the
// backward converts the effective-weight gradient into (dv, dg) in wn_grad_kernel.
struct WnRow {
  int w_off;          // flat offset of v[n][0]
  int g_idx;          // flat index of g[n]
  int ld;             // floats between rows of v
  int len;            // row length (kin + class columns)
  int kin;            // columns that go through the GEMM
  long long sh_off;   // bf16 shadow of the layer (-1: classifier row, fp32 copy only)
  int sh_rcap;
  int srow;           // shadow row
  long long aux_off;  // derived fp32: class-bias base of the layer, or the classifier's effective row
  int aux_ld;
};

// The classifier's hidden layers (dim_h_clf): u -> [Linear -> ELU] x nh -> linear_p.  Kept in device memory behind one
// pointer of the row kernels' view, which the plans without them do not read.
struct ClfView {
  int nh;
  int pin;        // input width of linear_p: the last hidden width
  C8Buf U;        // u with its ones column as the first hidden GEMM's operand ([z1 | z2f - z1 | 1] rows of DrVAE, written by
                  // clf_u_kernel; VFAE reads the z1 rows of Zdec)
  C8Buf H, D;     // last hidden activation (read by the logits row kernel) and its pre-activation gradient
  MBuf<float> dU; // DrVAE: [LNcap][clf_in] gradient of u, split into DZ1 / DZ2F by clf_du_kernel
};

struct MlpBlock {
  std::vector<Shadow> hidden;   // hidden[i]: layer i (ELU)
  Shadow head;                  // stacked (mu | lv) or interleaved (mu, sg) heads
  std::vector<int> widths;      // hidden widths
  bool class_aug = false;       // first layer input is [z, onehot(y)]
  std::vector<C8Buf> H;         // activations per hidden layer
  std::vector<C8Buf> dPre;      // pre-activation gradients per hidden layer
};

// ---------------------------------------------------------------------------------------------
// Device-visible view used by the row kernels
// ---------------------------------------------------------------------------------------------
// Scalars that may differ between ensemble members (drvae_set_member_hparams).  Every reader takes a base pointer and a
// model stride (DevView::member, EpiParams / DwaParams / AdamArgs adam + adam_ms): without a member table the stride
// is 0 and the base is the shared copy in StepDyn, so a table-less plan reads the same values as one without the
// feature; with a table the base is the plan's per-member array, expanded by set_dyn_kernel at the head of each step.
struct MemberScalars {
  float noise_std;
  float pertloss_rate, kl_qz2pz2_rate, yloss_rate;
  float log_prior[8];  // log prior_y
  AdamHyper adam;
};

struct StepScalars {
  float kl_min;
  float beta_pert;
  int training, add_noise;
  int gN, gNp, gNlab;  // global normalisers (0 = use local counts)
  int fused_adam;  // 1: the optimizer update happens inside the gradient kernels (drvae_train_step)
  MemberScalars mem;  // shared values of the per-member scalars
};

// Everything that changes from step to step.  Lives in device memory (one block per plan), written by
// set_dyn_kernel at the head of every launch sequence: kernels read it through DevView::dyn, so the
// sequence itself — grids, pointers, kernel arguments — is identical from step to step and can be
// replayed as a CUDA graph with only that one kernel node's arguments updated.
struct StepDyn {
  StepScalars s;
  float bc1;  // Adam bias correction 1 - beta1^t: a member's lr_bc1 is its lr / bc1 (set_dyn_kernel)
  unsigned int noise_step;
  unsigned long long noise_seed;
  long long row_offset;
  const long long* counts_dev;  // optional device {N, Np, Nlab} summed over the shards: overrides s.gN / gNp / gNlab
};

// Member table of a plan (drvae_set_member_hparams): set_dyn_kernel expands `table` (n entries, device) into `out`.
// n = 0: no table.
struct MemberExpand {
  const drvae_member_hparams_t* table;
  MemberScalars* out;
  int n;
};

struct DevView {
  int kind, X, Y, Z, Z3, L, N, Ncap;
  int model0;        // first ensemble member of this launch (a step may run sub-ranges of the ensemble as separate chains)
  int Xc;            // round_up(X, 16)
  int Zc, Z3c;       // chunk8 feature capacities of the latent buffers
  int Zs, Z3s;       // column of the logvar half in (mu | logvar) rows: round_up(Z, 16) / round_up(Z3, 16).  The two
                     // heads of a block are stacked in blocks of 16-aligned width, so an epilogue chunk or a 16-row
                     // stage of optimizer state never straddles the two weight tensors
  int clf_ld;        // floats between rows of the classifier weight
  int R0cap, LNcap, Rdcap, Fcap, Flcap;
  int has_pair, has_T, has_clf, has_fprop, clf_in;
  int need_grad;
  int clf_back_fused;  // 1: T_back computes the classifier's input gradient itself (no clf_back launch; DrVAE)
  int clf_split;     // 1: the classifier q(y|z1, z2f) runs as its own kernel (clf_fwd_kernel) off the main chain instead of inside T_post
  // batch (caller memory)
  MBuf<const float> x1, x2;
  MBuf<const int> y, has_x2, has_y;
  MBuf<const int> row_index;  // optional [N] per model: the batch is rows row_index[i] of a device-resident dataset
  // ε (row indexed)
  MBuf<const float> eps_x1, eps_x2, eps_z1, eps_z2, eps_z2f, eps_z3;
  // own_noise: the input noise of x1 / x2 is drawn inside prep_kernel (same Philox keys as the ε
  // generator, segments 0 and 1) instead of being written to and read back from the ε block
  int own_noise;
  // row maps
  MBuf<int> counts;   // CNT_*
  MBuf<float> coefs;  // COEF_*
  MBuf<int> pair_of, row_of_pair, ebase, lab, ycls, e_row, e_jj, e_cls_full;
  // activations
  MBuf<float4> tgt4;  // fp32 targets, chunk4: [Xc/4][R0cap] float4
  C8Buf Ain;        // [Xc/8][R0cap][8]
  MBuf<float> Q;    // [R0cap][2 Zs] (mu1 | lv1) rows < N, (mu2 | lv2) rows N + p; logvar at column Zs
  MBuf<float> Z1f;  // [LNcap][Z]
  C8Buf Zdec;       // rows: z1 (L*N) | z2 (L*Np) | z2f (L*Np)
  C8Buf Z1e;        // eval-ordered copies of z1
  MBuf<float> PT;   // [LNcap][2 Zs] (p_mu | p_lv) of p(z2|z1)
  MBuf<float> Z2Ff; // [LNcap][Z]
  MBuf<float> QY;   // [LNcap][Y]
  MBuf<float> Q3;   // [Fcap][2 Z3s]
  C8Buf Z3b;        // [Z3c/8][Fcap][8]
  MBuf<float> PZ1;  // [Fcap][2 Zs]
  // per-row loss terms
  MBuf<float> klq_row;   // [R0cap]  PVAE prior KLs
  MBuf<float> klz2_row;  // [LNcap]
  MBuf<float> yl_row;    // [LNcap]
  MBuf<float> ycat_row;  // [LNcap]
  MBuf<float> kfp_row;   // [Fcap]   fb(KL3) + fb(KLp) per evaluation
  MBuf<float> kfpw_row;  // [Fcap]   weighted by q(y)
  MBuf<float> dec_part;  // [dec_tiles][Rdcap]
  int dec_tiles;
  // backward
  C8Buf dY9, dY7, dYT, dY2;
  MBuf<float> dQ1e;    // [Fcap][2 Zs]
  MBuf<float> dQ2;     // [Ncap][2 Zs]
  MBuf<float> dZ3;     // [Fcap][Z3]
  MBuf<float> dZ1e;    // [Fcap][Z]
  MBuf<float> dZdec;   // [Rdcap][Z]
  MBuf<float> dZ1T;    // [LNcap][Z]
  MBuf<float> DZ1;     // [LNcap][Z]
  MBuf<float> DZ2F;    // [LNcap][Z]
  MBuf<float> dlogit;  // [LNcap][Y]
  MBuf<float> clf_part; // [clf_splits][Y][clf_in + 1]
  int clf_splits;
  MBuf<float> loss_part;  // [loss_slices][8] partial sums of the loss terms
  int loss_slices;
  // parameters
  MBuf<float> params, grads, adam_m, adam_v;
  int clf_w_off, clf_b_off;
  MBuf<const float> clf_w;  // classifier weights as the kernels read them: the parameters, or the
                            // effective (weight-normalised) copy in the derived arena
  MBuf<float> losses;  // [8]
  const StepDyn* dyn;  // per-step scalars (device memory)
  const MemberScalars* mem;  // per-member scalars of global model m: mem[m * mem_stride] (stride 0: the copy in dyn)
  int mem_stride;
  __host__ __device__ __forceinline__ const MemberScalars& member(int m) const { return mem[(long long)m * mem_stride]; }
  SampleView* sview_dev;  // device copy of the sampling epilogue's view (written by rowmap_kernel; null: not used)
  unsigned long long* trace;  // kernel trace buffer (null: off) and this launch's slot
  int trace_id;
  const ClfView* clf;  // classifier hidden layers (device memory); null: linear_p reads u itself
};

constexpr int CLF_SPLITS = 32;       // row splits of the classifier weight gradient (ensemble-sized batches)
constexpr int CLF_SPLITS_MAX = 512;  // ... for large single-model minibatches
constexpr int LOSS_SLICES_MAX = 64;  // row slices of the loss reduction
constexpr int MAXY = 8;   // classes
constexpr int MAXJ = 8;   // latent dim <= 32 * MAXJ

}  // namespace drvae
