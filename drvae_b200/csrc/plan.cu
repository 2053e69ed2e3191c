// Plan construction (parameter layout, weight shadows, workspace) and the step executor: the
// host side of the C ABI in include/drvae_b200.h.  One launch sequence trains every member of
// the ensemble; all row counts are read on the device, so the sequence is fixed per (plan, N).
#include <math.h>
#include <string.h>

#include <algorithm>
#include <functional>

#include <map>
#include <string>
#include <vector>

#include "errors.h"
#include "dp_peer.cuh"
#include "dwadam.cuh"
#include "gemm.cuh"
#include "infer_f32.cuh"
#include "optim.cuh"
#include "plan.h"
#include "rowops.cuh"
#include "stepk.cuh"

using namespace drvae;

namespace {

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }
inline int cdiv(int a, int b) { return (a + b - 1) / b; }

struct Tiling {
  int BN, tiles, cap;
};
// N tiling of a feature dimension: tiles of equal width (multiple of 16, <= 256).
Tiling tile_cap(int n) {
  const int n16 = round_up(n, 16);
  Tiling t;
  t.tiles = cdiv(n16, 256);
  t.BN = round_up(cdiv(n16, t.tiles), 16);
  t.cap = t.BN * t.tiles;
  return t;
}

struct BufRec {
  size_t off;       // byte offset in the arena
  size_t ms_bytes;  // bytes between models
  size_t bytes;     // used bytes per model
  int rcap, fcap;
};

}  // namespace

struct drvae_plan {
  drvae_arch_t arch;
  int E;
  int X, Y, Z, Z3, L, Ncap;
  int has_pair, has_T, has_clf, has_fprop, clf_in;
  int clf_nh = 0, clf_pin = 0;  // classifier hidden layers (dim_h_clf) and the input width of linear_p
  // parameters
  std::vector<ParamInfo> tensors;
  std::vector<Seg> segs;
  Seg* d_segs = nullptr;
  std::vector<int> h_tabs;  // gradient-epilogue tables of every weight (see make_shadow)
  int* d_tabs = nullptr;
  bool wn = false;            // layers.WeightNormLinear instead of nn.Linear
  std::vector<WnRow> wn_rows;
  WnRow* d_wn_rows = nullptr;
  long long clf_eff_off = -1;  // derived offset of the classifier's effective weights (weight norm only)
  int P = 0;
  long long T_range[2] = {0, 0};  // (offset, count) of the decoder_z2Fz1 parameters
  int clf_w_off = -1, clf_b_off = -1;
  // shadows
  long long shadow_elems = 0;   // bf16 per model
  long long derived_elems = 0;  // fp32 per model
  MlpBlock enc, dec, z3b, dz1b;
  MlpBlock clfb;  // classifier hidden layers (no head: linear_p stays an fp32 row kernel)
  ClfView clfv{};  // ... their buffers, and the device copy the row kernels read (DevView::clf)
  ClfView* d_clfv = nullptr;
  Shadow Tsh;
  int dec_hb = 0;
  // workspace
  size_t arena_bytes = 0;
  uint8_t* arena = nullptr;
  std::map<std::string, BufRec> bufs;
  C8Buf dY5;  // decoder head gradient
  MBuf<float> eps_own;
  drvae_eps_layout_t epsl;
  MBuf<bf16> shadow;
  MBuf<float> derived;
  DevView view;  // static part
  DebugWord* dbg = nullptr;
  // bound state
  float *params = nullptr, *adam_m = nullptr, *adam_v = nullptr, *grads = nullptr;
  int gemm_impl = GEMM_IMPL_TC;
  int act = DRVAE_ACT_ELU;  // hidden-layer activation of every MLP (drvae_set_activation)
  long long launches = 0;
  bool shadows_valid = false;
  // per-step scalars in device memory + CUDA-graph replay of the launch sequence (see step_entry)
  StepDyn* d_dyn = nullptr;
  // member table (drvae_set_member_hparams): device copy of the caller's table, its per-step expansion, and the pinned
  // staging the copy is made from (member_ev: the last copy out of it)
  bool member_table = false;
  drvae_member_hparams_t* d_member_hp = nullptr;
  MemberScalars* d_member = nullptr;
  drvae_member_hparams_t* h_member_stage = nullptr;
  cudaEvent_t member_ev = nullptr;
  bool graph_enabled = true;
  struct GraphEntry {
    int seen = 0;
    cudaGraph_t graph = nullptr;  // kept alive: node handles used for parameter updates belong to it
    cudaGraphExec_t exec = nullptr;
    cudaGraphNode_t dyn_node = nullptr;
    cudaKernelNodeParams dyn_params{};
    long long launches = 0;
    long long last_use = 0;
  };
  std::map<std::vector<long long>, GraphEntry> graphs;
  long long graph_clock = 0;
  long long graph_replays = 0;
  long long graph_failures = 0;  // capture / instantiation failures (those combinations run as plain launches)
  // streams and events of the step schedule (see run_step): the plan's high-priority main stream, the low-priority side
  // stream of the label-dependent branch, and a low-priority stream for the early part of the grouped dW+Adam launch
  cudaStream_t s_main = nullptr, s_side = nullptr, s_dwa = nullptr;
  struct StepEvents {
    cudaEvent_t begin = nullptr, fork = nullptr, qy = nullptr, side_fwd = nullptr, side_bwd = nullptr, noise = nullptr, eps = nullptr,
                clf = nullptr, kfp = nullptr, end = nullptr, side_end = nullptr, dw = nullptr, dw_end = nullptr, dwa = nullptr,
                dwa_end = nullptr;
    static constexpr int N = 15;
    cudaEvent_t* all() { return &begin; }  // N consecutive events
  } ev;
  long long side_delay_cycles = 0;  // test knob (drvae_debug_side_delay): spin on the side stream before pz1_post
  // gradient buckets (data-parallel overlap): contiguous parameter ranges in backward completion order
  std::vector<std::pair<long long, long long>> buckets;  // (offset, count)
  std::vector<cudaEvent_t> bucket_ev;
  // grouped weight-gradient + Adam launch (dwadam.cuh): layer table and tensor maps in device memory, rebuilt by bind
  std::vector<DwaLayer> dwa_layers;
  DwaLayer* d_dwa_layers = nullptr;
  DwaMaps* d_dwa_maps = nullptr;
  int dwa_tiles = 0;
  bool dwa_ok = false;       // every layer fits the kernel's layout conditions and the state is bound
  unsigned long long* d_dwa_stats = nullptr;  // drvae_debug_dwa_stats
  // Early part of the grouped launch: the decoder heads (half of the optimizer state) have all their inputs once the
  // decoder's dX GEMM has run; their tiles start then, on dwa_early_sms SMs, next to the latency-bound rest of the
  // backward chain (whose persistent GEMMs are capped to the remaining SMs).  0: one launch at the end.
  int dwa_early_tiles = 0;   // tiles of the first layer when that layer is the decoder head block
  int dwa_early_sms = 92;    // DRVAE_B200_DWA_EARLY_SMS (measured on two boxes: 0.939 -> 0.918 ms at 84, 0.953 -> 0.943 at 100; 72 and 116+ lose)
  // persistent step kernel (stepk.cuh): the forward + input-gradient chain as one cooperative launch
  bool stepk_enabled = false;          // drvae_set_step_kernel / DRVAE_B200_STEPK (measured slower than the graph of launches: profiles/r02_experiments.md)
  bool stepk_unsupported = false;      // a recorded sequence did not fit the kernel's tables: this plan launches kernel by kernel
  unsigned int* d_stepk_bar = nullptr; // {arrival count, generation}
  long long stepk_launches = 0;
  // data-parallel exchange over peer memory (dp_peer.cuh): attached by drvae_dp_attach
  bool dp_on = false;
  DpPeers dp{};
  long long* dp_counts = nullptr;  // int64 [3]: batch-global {N, Np, Nlab} of the current step
  // fp32 inference path (infer_f32.cuh): on by default (exact thresholded predictions); scratch allocated on first use
  bool infer_fp32 = true;
  float* f32ws = nullptr;
  size_t f32ws_floats = 0;
  // kernel trace (drvae_trace_begin / _end): device slots {first CTA start, last CTA end} per launch, tags on the host
  unsigned long long* d_trace = nullptr;
  int trace_cap = 0, trace_next = 0;
  bool trace_on = false, trace_saved_graph = true;
  std::vector<std::string> trace_tags;
  // optional per-launch event timing (bench.py / profiles)
  bool prof_on = false;
  std::vector<cudaEvent_t> prof_ev;
  std::vector<std::string> prof_tags;
  size_t prof_used = 0;
  std::map<std::string, std::pair<long long, double>> prof_acc;  // tag -> (launches, ms)
};

namespace {

// ---------------------------------------------------------------------------------------------
// parameter layout
// ---------------------------------------------------------------------------------------------
int add_tensor(drvae_plan* pl, const std::string& name, int rows, int cols) {
  ParamInfo t;
  t.name = name;
  t.rows = rows;
  t.cols = cols;
  // every tensor starts on a 16-byte boundary of the flat vector (TMA boxes of the grouped dW+Adam launch address
  // the optimizer state from 16-byte aligned tensor starts); the padding elements are zero parameters with zero
  // gradients and stay zero
  pl->P = round_up(pl->P, 4);
  t.off = pl->P;
  // matrix rows are 16-byte aligned as well (row stride = cols rounded up to 4 floats): the optimizer state of a
  // weight tile can then be moved by TMA tensor loads / stores (global strides must be multiples of 16 bytes) and
  // every layer takes the 16-byte epilogue paths.  Padding elements behave like the padding between tensors.
  t.ld = cols > 0 ? round_up(cols, 4) : 1;
  pl->P += rows * t.ld;
  pl->tensors.push_back(t);
  return (int)pl->tensors.size() - 1;
}

void add_seg_plain(drvae_plan* pl, int tid) {
  const ParamInfo& t = pl->tensors[tid];
  Seg s{};
  s.off = t.off;
  s.rows = t.rows;
  s.cols = t.cols > 0 ? t.cols : 1;
  s.ld = t.ld;
  s.kind = SEG_PLAIN;
  s.wn_g_off = -1;
  s.ilv_block = s.ilv_stride = 1 << 30;
  pl->segs.push_back(s);
}

// Allocate shadow storage + derived bias for a GEMM weight made of `ntens` reference tensors.
Shadow make_shadow(drvae_plan* pl, int ntens, const int* w_tid, const int* b_tid, int rows_each, int kin, int class_cols,
                   int ilv_block, int ilv_stride, int BN, int tiles_n, const float* bias_const, const int* g_tid = nullptr) {
  Shadow sh{};
  sh.g_off[0] = sh.g_off[1] = -1;
  sh.ntens = ntens;
  sh.kin = kin;
  sh.kaug = kin + 1 + class_cols;
  sh.kc = round_up(sh.kaug, 16);
  sh.BN = BN;
  sh.tiles_n = tiles_n;
  sh.rcap = BN * tiles_n;
  Tiling tx = tile_cap(kin);
  sh.BNx = tx.BN;
  sh.tiles_nx = tx.tiles;
  sh.ilv_block = ilv_block;
  sh.ilv_stride = ilv_stride;
  sh.ld = round_up(kin + class_cols, 4);
  sh.off = pl->shadow_elems;
  pl->shadow_elems += (long long)(sh.kc / 8) * sh.rcap * 8;
  sh.bias_off = pl->derived_elems;
  pl->derived_elems += sh.rcap;
  sh.clsb_off = -1;
  if (class_cols > 0) {
    sh.clsb_off = pl->derived_elems;
    pl->derived_elems += (long long)class_cols * sh.rcap;
  }
  int max_srow = 0;
  for (int w = 0; w < ntens; ++w) {
    const ParamInfo& wt = pl->tensors[w_tid[w]];
    const ParamInfo& bt = pl->tensors[b_tid[w]];
    sh.w_off[w] = wt.off;
    sh.b_off[w] = bt.off;
    sh.rows_each[w] = rows_each;
    sh.bias_const[w] = bias_const ? bias_const[w] : 0.f;
    Seg s{};
    s.off = wt.off;
    s.rows = wt.rows;
    s.cols = wt.cols;
    s.ld = wt.ld;
    s.kind = SEG_W;
    s.sh_off = sh.off;
    s.sh_rcap = sh.rcap;
    s.kmain = kin;
    s.which = w;
    s.ilv_block = ilv_block;
    s.ilv_stride = ilv_stride;
    s.clsb_off = sh.clsb_off;
    s.clsb_ld = sh.rcap;
    s.wn_g_off = -1;
    if (g_tid) {
      sh.g_off[w] = pl->tensors[g_tid[w]].off;
      s.wn_g_off = sh.g_off[w];
      add_seg_plain(pl, g_tid[w]);
    }
    pl->segs.push_back(s);
    Seg b{};
    b.off = bt.off;
    b.rows = bt.rows;
    b.cols = 1;
    b.ld = 1;
    b.kind = SEG_B;
    b.which = w;
    b.ilv_block = ilv_block;
    b.ilv_stride = ilv_stride;
    b.bias_off = sh.bias_off;
    b.bias_const = bias_const ? bias_const[w] : 0.f;
    b.wn_g_off = -1;
    pl->segs.push_back(b);
    const int n = rows_each - 1;
    const int srow = (n / ilv_block) * ilv_stride + w * ilv_block + (n % ilv_block);
    if (srow > max_srow) max_srow = srow;
  }
  sh.nout_total = max_srow + 1;
  // gradient-epilogue tables, indexed by shadow row s: flat offset of W[n(s)][0] (-1: padding),
  // flat offset of b[n(s)], constant folded into the derived bias
  sh.tab_off = (long long)pl->h_tabs.size();
  pl->h_tabs.resize(pl->h_tabs.size() + 3 * (size_t)sh.rcap, -1);
  int* tw = pl->h_tabs.data() + sh.tab_off;
  for (int srow = 0; srow < sh.rcap; ++srow) {
    const int blk = srow / ilv_stride, rem = srow % ilv_stride;
    const int which = rem / ilv_block, n = blk * ilv_block + rem % ilv_block;
    if (which < ntens && n < rows_each) {
      tw[srow] = sh.w_off[which] + n * sh.ld;
      tw[sh.rcap + srow] = sh.b_off[which] + n;
      float c = sh.bias_const[which];
      memcpy(&tw[2 * sh.rcap + srow], &c, sizeof(float));
      if (sh.g_off[which] >= 0) {
        WnRow r{};
        r.w_off = sh.w_off[which] + n * sh.ld;
        r.g_idx = sh.g_off[which] + n;
        r.ld = sh.ld;
        r.len = kin + class_cols;
        r.kin = kin;
        r.sh_off = sh.off;
        r.sh_rcap = sh.rcap;
        r.srow = srow;
        r.aux_off = sh.clsb_off;
        r.aux_ld = sh.rcap;
        pl->wn_rows.push_back(r);
      }
    }
  }
  return sh;
}

// blocks.MLP: `nh` Linear + ELU layers <prefix>.nnet.model.linear{1..nh}; returns the width of the last one.
int build_hidden(drvae_plan* pl, MlpBlock& blk, const std::string& prefix, int in_dim, int class_cols, int nh, const int* widths) {
  blk.class_aug = class_cols > 0;
  int prev = in_dim;
  for (int i = 0; i < nh; ++i) {
    char nm[160];
    snprintf(nm, sizeof(nm), "%s.nnet.model.linear%d", prefix.c_str(), i + 1);
    const int cc = (i == 0) ? class_cols : 0;
    int w = add_tensor(pl, std::string(nm) + ".weight", widths[i], prev + cc);
    int b = add_tensor(pl, std::string(nm) + ".bias", widths[i], 0);
    int g = pl->wn ? add_tensor(pl, std::string(nm) + ".g", widths[i], 0) : -1;
    Tiling t = tile_cap(widths[i] + 1);  // + the ones column the next layer's dW reads
    blk.hidden.push_back(
        make_shadow(pl, 1, &w, &b, widths[i], prev, cc, 1 << 30, 1 << 30, t.BN, t.tiles, nullptr, pl->wn ? &g : nullptr));
    blk.widths.push_back(widths[i]);
    prev = widths[i];
  }
  return prev;
}

// blocks.DiagGaussianModule / DiagGaussianSigmaModule: hidden MLP + two heads.
void build_gauss_block(drvae_plan* pl, MlpBlock& blk, const std::string& prefix, int in_dim, int class_cols, int nh,
                       const int* widths, int out_dim, bool sigma_heads) {
  const int prev = build_hidden(pl, blk, prefix, in_dim, class_cols, nh, widths);
  int wt[2], bt[2], gt[2] = {-1, -1};
  const char* second = sigma_heads ? "sg" : "lv";
  const std::string heads[2] = {prefix + ".encoder_mu.linear_mu", prefix + ".encoder_" + second + ".linear_" + second};
  for (int w = 0; w < 2; ++w) {
    wt[w] = add_tensor(pl, heads[w] + ".weight", out_dim, prev);
    bt[w] = add_tensor(pl, heads[w] + ".bias", out_dim, 0);
    if (pl->wn) gt[w] = add_tensor(pl, heads[w] + ".g", out_dim, 0);
  }
  if (!sigma_heads) {
    const float bc[2] = {0.f, -2.f};  // logvar = lin(h) - 2  (blocks.py:296)
    const int os = round_up(out_dim, 16);  // (mu | logvar) stacked in 16-aligned blocks (DevView::Zs)
    Tiling t = tile_cap(2 * os);
    blk.head = make_shadow(pl, 2, wt, bt, out_dim, prev, 0, os, 2 * os, t.BN, t.tiles, bc, pl->wn ? gt : nullptr);
  } else {
    const int hb = std::min(128, round_up(out_dim, 16));
    pl->dec_hb = hb;
    blk.head = make_shadow(pl, 2, wt, bt, out_dim, prev, 0, hb, 2 * hb, 2 * hb, cdiv(out_dim, hb), nullptr, pl->wn ? gt : nullptr);
  }
}

struct ArenaBuilder {
  size_t total = 0;
  int E;
  std::map<std::string, BufRec>* bufs;
  BufRec take(const std::string& name, size_t bytes_per_model, int rcap = 0, int fcap = 0) {
    BufRec r;
    r.off = total;
    r.bytes = bytes_per_model;
    r.ms_bytes = (bytes_per_model + 255) / 256 * 256;
    r.rcap = rcap;
    r.fcap = fcap;
    total += r.ms_bytes * E;
    (*bufs)[name] = r;
    return r;
  }
};

template <class T>
MBuf<T> mbuf_of(drvae_plan* pl, const BufRec& r) {
  MBuf<T> b;
  b.p = reinterpret_cast<T*>(pl->arena + r.off);
  b.ms = (long long)(r.ms_bytes / sizeof(T));
  return b;
}
C8Buf c8_of(drvae_plan* pl, const BufRec& r) {
  C8Buf b;
  b.p = reinterpret_cast<bf16*>(pl->arena + r.off);
  b.ms = (long long)(r.ms_bytes / sizeof(bf16));
  b.rcap = r.rcap;
  b.fcap = r.fcap;
  return b;
}

}  // namespace

namespace {
void drop_graphs(drvae_plan* pl) {
  for (auto& kv : pl->graphs) {
    if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
    if (kv.second.graph) cudaGraphDestroy(kv.second.graph);
  }
  pl->graphs.clear();
}
}  // namespace

// =============================================================================================
// plan creation
// =============================================================================================
extern "C" int drvae_plan_create(const drvae_arch_t* a, int n_models, drvae_plan_t** out) {
  return drvae_plan_create_clf(a, 0, nullptr, n_models, out);
}

extern "C" int drvae_plan_create_clf(const drvae_arch_t* a, int n_clf, const int* clf_hidden, int n_models, drvae_plan_t** out) {
  if (!a || !out) return set_error("drvae_plan_create: null argument");
  if (n_models < 1) return set_error("drvae_plan_create: n_models must be >= 1");
  // the Philox counter has 20 bits for the model and 8 for the MC sample (drvae_noise_t): beyond them two models or two
  // samples would draw the same normals
  if (n_models > DRVAE_MAX_MODELS) return set_error("drvae_plan_create: n_models must be <= 1048576 (2^20)");
  if (a->kind < 0 || a->kind > 2) return set_error("drvae_plan_create: unknown model kind");
  if (a->dim_x < 1 || a->dim_z1 < 1 || a->L < 1 || a->max_batch < 1) return set_error("drvae_plan_create: bad dimensions");
  if (a->L > DRVAE_MAX_L) return set_error("drvae_plan_create: L must be <= 256 Monte-Carlo samples");
  if (a->dim_z1 > 32 * MAXJ) return set_error("drvae_plan_create: dim_z1 > 256 is not supported");
  if (a->kind != DRVAE_KIND_PVAE && (a->dim_y < 2 || a->dim_y > MAXY)) return set_error("drvae_plan_create: dim_y must be in [2, 8]");
  if (a->kind != DRVAE_KIND_PVAE && (a->dim_z3 < 1 || a->dim_z3 > 32 * MAXJ)) return set_error("drvae_plan_create: dim_z3 must be in [1, 256]");
  if (a->n_enc_z1 < 1 || a->n_enc_z1 > DRVAE_MAX_HIDDEN || a->n_dec_x < 1 || a->n_dec_x > DRVAE_MAX_HIDDEN)
    return set_error("drvae_plan_create: enc_z1 / dec_x need between 1 and 4 hidden layers");
  if (a->kind != DRVAE_KIND_PVAE &&
      (a->n_enc_z3 < 1 || a->n_enc_z3 > DRVAE_MAX_HIDDEN || a->n_dec_z1 < 1 || a->n_dec_z1 > DRVAE_MAX_HIDDEN))
    return set_error("drvae_plan_create: enc_z3 / dec_z1 need between 1 and 4 hidden layers");
  if (n_clf < 0 || n_clf > DRVAE_MAX_HIDDEN) return set_error("drvae_plan_create_clf: n_clf must be in [0, 4]");
  if (n_clf > 0 && a->kind == DRVAE_KIND_PVAE)
    return set_error("drvae_plan_create_clf: PVAE has no classifier, n_clf must be 0");
  if (n_clf > 0 && !clf_hidden) return set_error("drvae_plan_create_clf: clf_hidden is null");
  for (int i = 0; i < n_clf; ++i)
    if (clf_hidden[i] < 1 || clf_hidden[i] > DRVAE_MAX_CLF_WIDTH)
      return set_error("drvae_plan_create_clf: classifier hidden widths must be in [1, 4096]");

  drvae_plan* pl = new drvae_plan();
  pl->arch = *a;
  pl->wn = a->weight_norm != 0;
  pl->E = n_models;
  pl->X = a->dim_x;
  pl->Y = (a->kind == DRVAE_KIND_PVAE) ? 1 : a->dim_y;
  pl->Z = a->dim_z1;
  pl->Z3 = (a->kind == DRVAE_KIND_PVAE) ? 1 : a->dim_z3;
  pl->L = a->L;
  pl->Ncap = a->max_batch;
  pl->has_pair = a->kind != DRVAE_KIND_VFAE;
  pl->has_T = a->kind != DRVAE_KIND_VFAE;
  pl->has_clf = a->kind != DRVAE_KIND_PVAE;
  pl->has_fprop = a->kind != DRVAE_KIND_PVAE;
  pl->clf_in = (a->kind == DRVAE_KIND_DRVAE) ? 2 * pl->Z : pl->Z;
  pl->clf_nh = n_clf;
  pl->clf_pin = n_clf > 0 ? clf_hidden[n_clf - 1] : pl->clf_in;
  const int X = pl->X, Y = pl->Y, Z = pl->Z, Z3 = pl->Z3, L = pl->L, E = pl->E;

  // ---- parameters in the reference's state_dict order (SURVEY.md Appendix C) ----
  int p0 = pl->P;
  long long r_enc[2], r_T[2] = {0, 0}, r_clf[2] = {0, 0}, r_z3[2] = {0, 0}, r_dz1[2] = {0, 0}, r_dec[2];
  build_gauss_block(pl, pl->enc, "encoder_z1", X, 0, a->n_enc_z1, a->enc_z1, Z, false);
  r_enc[0] = p0, r_enc[1] = pl->P - p0, p0 = pl->P;
  if (pl->has_T) {
    // DiagGaussianModuleLinear (blocks.py:304-361): W_mu, bias_mu are bare Parameters
    int wt[2], bt[2];
    wt[0] = add_tensor(pl, "decoder_z2Fz1.W_mu", Z, Z);
    bt[0] = add_tensor(pl, "decoder_z2Fz1.bias_mu", Z, 0);
    wt[1] = add_tensor(pl, "decoder_z2Fz1.encoder_lv.linear_lv.weight", Z, Z);
    bt[1] = add_tensor(pl, "decoder_z2Fz1.encoder_lv.linear_lv.bias", Z, 0);
    const float bc[2] = {0.f, -2.f};
    const int Zs = round_up(Z, 16);
    Tiling t = tile_cap(2 * Zs);
    pl->Tsh = make_shadow(pl, 2, wt, bt, Z, Z, 0, Zs, 2 * Zs, t.BN, t.tiles, bc);
    r_T[0] = p0, r_T[1] = pl->P - p0, p0 = pl->P;
    pl->T_range[0] = r_T[0], pl->T_range[1] = r_T[1];
  }
  if (pl->has_clf) {
    // CategoricalDecoder (blocks.py:456-463): its MLP (nnet) first, then linear_p
    build_hidden(pl, pl->clfb, "encoder_y", pl->clf_in, 0, pl->clf_nh, clf_hidden);
    int w = add_tensor(pl, "encoder_y.decoder_p.linear_p.weight", Y, pl->clf_pin);
    int b = add_tensor(pl, "encoder_y.decoder_p.linear_p.bias", Y, 0);
    pl->clf_w_off = pl->tensors[w].off;
    pl->clf_b_off = pl->tensors[b].off;
    add_seg_plain(pl, w);
    add_seg_plain(pl, b);
    if (pl->wn) {
      int g = add_tensor(pl, "encoder_y.decoder_p.linear_p.g", Y, 0);
      add_seg_plain(pl, g);
      pl->clf_eff_off = pl->derived_elems;
      pl->derived_elems += round_up(Y * pl->tensors[w].ld, 64);
      for (int n = 0; n < Y; ++n) {
        WnRow r{};
        r.w_off = pl->clf_w_off + n * pl->tensors[w].ld;
        r.g_idx = pl->tensors[g].off + n;
        r.ld = pl->tensors[w].ld;
        r.len = r.kin = pl->clf_pin;
        r.sh_off = -1;
        r.aux_off = pl->clf_eff_off + (long long)n * pl->tensors[w].ld;
        pl->wn_rows.push_back(r);
      }
    }
    r_clf[0] = p0, r_clf[1] = pl->P - p0, p0 = pl->P;
  }
  if (pl->has_fprop) {
    const char* top = (a->kind == DRVAE_KIND_DRVAE) ? "encoder_z3" : "encoder_z2";
    build_gauss_block(pl, pl->z3b, top, Z, Y, a->n_enc_z3, a->enc_z3, Z3, false);
    r_z3[0] = p0, r_z3[1] = pl->P - p0, p0 = pl->P;
    build_gauss_block(pl, pl->dz1b, "decoder_z1", Z3, Y, a->n_dec_z1, a->dec_z1, Z, false);
    r_dz1[0] = p0, r_dz1[1] = pl->P - p0, p0 = pl->P;
  }
  build_gauss_block(pl, pl->dec, "decoder_x", Z, 0, a->n_dec_x, a->dec_x, X, true);
  pl->P = round_up(pl->P, 4);  // model stride of the flat vectors: 16-byte aligned
  r_dec[0] = p0, r_dec[1] = pl->P - p0;
  // backward completes the blocks in this order (run_step)
  if (pl->has_fprop) {
    pl->buckets.push_back({r_dz1[0], r_dz1[1]});
    pl->buckets.push_back({r_z3[0], r_z3[1]});
  }
  pl->buckets.push_back({r_dec[0], r_dec[1]});
  if (pl->has_clf) pl->buckets.push_back({r_clf[0], r_clf[1]});
  if (pl->has_T) pl->buckets.push_back({r_T[0], r_T[1]});
  pl->buckets.push_back({r_enc[0], r_enc[1]});
  std::sort(pl->segs.begin(), pl->segs.end(), [](const Seg& x, const Seg& y) { return x.off < y.off; });

  // ---- workspace ----
  const int Ncap = pl->Ncap;
  const int R0cap = round_up((pl->has_pair ? 2 : 1) * Ncap, 128);
  const int LNcap = round_up(L * Ncap, 128);
  const int Rdcap = round_up((pl->has_pair ? 3 : 1) * L * Ncap, 128) + 128;  // +1 tile: inference reads H at row offset N
  const int Flcap = pl->has_fprop ? Y * Ncap : 0;
  const int Fcap = round_up(std::max(1, L * Flcap), 128);
  // feature capacities of the GEMM input buffers: features + ones column (+ one-hot class columns)
  const int Xc = round_up(X + 1, 16);
  const int Zc = round_up(Z + 1 + (pl->has_fprop ? Y : 0), 16), Z3c = round_up(Z3 + 1 + Y, 16);
  const int Zs = round_up(Z, 16), Z3s = round_up(Z3, 16);

  ArenaBuilder ab;
  ab.E = E;
  ab.bufs = &pl->bufs;
  auto F32 = [&](const char* n, size_t elems) { return ab.take(n, elems * 4); };
  auto I32 = [&](const char* n, size_t elems) { return ab.take(n, elems * 4); };
  auto C8 = [&](const std::string& n, int rcap, int fcap) { return ab.take(n, (size_t)rcap * fcap * 2, rcap, fcap); };

  BufRec r_shadow = ab.take("shadow", (size_t)pl->shadow_elems * 2);
  BufRec r_derived = F32("derived", pl->derived_elems);
  // ε block
  drvae_eps_layout_t& el = pl->epsl;
  el.off_x1 = 0;
  el.off_x2 = el.off_x1 + (long long)Ncap * X;
  el.off_z1 = el.off_x2 + (long long)Ncap * X;
  el.off_z2 = el.off_z1 + (long long)L * Ncap * Z;
  el.off_z2f = el.off_z2 + (long long)L * Ncap * Z;
  el.off_z3 = el.off_z2f + (long long)L * Ncap * Z;
  el.total = el.off_z3 + (long long)L * Ncap * Y * Z3;
  BufRec r_eps = F32("eps", el.total);
  BufRec r_counts = I32("counts", CNT_SIZE), r_coefs = F32("coefs", COEF_SIZE);
  BufRec r_pair_of = I32("pair_of", Ncap), r_row_of_pair = I32("row_of_pair", Ncap), r_ebase = I32("ebase", Ncap);
  BufRec r_lab = I32("lab", Ncap), r_ycls = I32("ycls", Ncap), r_e_row = I32("e_row", std::max(1, Flcap));
  BufRec r_e_jj = I32("e_jj", std::max(1, Flcap)), r_e_cls = I32("e_cls_full", Fcap);
  BufRec r_tgt = F32("tgt4", (size_t)R0cap * Xc);
  BufRec r_Ain = C8("Ain", R0cap, Xc);
  BufRec r_Q = F32("Q", (size_t)R0cap * 2 * Zs), r_Z1f = F32("Z1f", (size_t)LNcap * Z);
  BufRec r_Zdec = C8("Zdec", Rdcap, Zc), r_Z1e = C8("Z1e", Fcap, Zc);
  BufRec r_PT = F32("PT", (size_t)LNcap * 2 * Zs), r_Z2Ff = F32("Z2Ff", (size_t)LNcap * Z);
  BufRec r_QY = F32("QY", (size_t)LNcap * Y), r_Q3 = F32("Q3", (size_t)Fcap * 2 * Z3s);
  BufRec r_Z3b = C8("Z3b", Fcap, Z3c), r_PZ1 = F32("PZ1", (size_t)Fcap * 2 * Zs);
  BufRec r_klq = F32("klq_row", R0cap), r_klz2 = F32("klz2_row", LNcap), r_yl = F32("yl_row", LNcap);
  BufRec r_ycat = F32("ycat_row", LNcap), r_kfp = F32("kfp_row", Fcap), r_kfpw = F32("kfpw_row", Fcap);
  const int dec_tiles = pl->dec.head.tiles_n * EPI_GROUPS;
  BufRec r_part = F32("dec_part", (size_t)dec_tiles * Rdcap);
  BufRec r_dY5 = C8("dY5", Rdcap, pl->dec.head.rcap);
  BufRec r_dY9 = C8("dY9", Fcap, pl->has_fprop ? pl->dz1b.head.rcap : 16);
  BufRec r_dY7 = C8("dY7", Fcap, pl->has_fprop ? pl->z3b.head.rcap : 16);
  BufRec r_dYT = C8("dYT", LNcap, pl->has_T ? pl->Tsh.rcap : 16);
  BufRec r_dY2 = C8("dY2", R0cap, pl->enc.head.rcap);
  BufRec r_dQ1e = F32("dQ1e", (size_t)Fcap * 2 * Zs), r_dQ2 = F32("dQ2", (size_t)Ncap * 2 * Zs);
  BufRec r_dZ3 = F32("dZ3", (size_t)Fcap * Z3), r_dZ1e = F32("dZ1e", (size_t)Fcap * Z);
  BufRec r_dZdec = F32("dZdec", (size_t)Rdcap * Z), r_dZ1T = F32("dZ1T", (size_t)LNcap * Z);
  BufRec r_DZ1 = F32("DZ1", (size_t)LNcap * Z), r_DZ2F = F32("DZ2F", (size_t)LNcap * Z);
  BufRec r_dlogit = F32("dlogit", (size_t)LNcap * Y);
  BufRec r_clfp = F32("clf_part", (size_t)CLF_SPLITS_MAX * Y * (std::max(pl->clf_in, pl->clf_pin) + 1));
  BufRec r_lossp = F32("loss_part", (size_t)LOSS_SLICES_MAX * 8);
  BufRec r_losses = F32("losses", 8);
  // per-block activations
  struct BlkAlloc {
    MlpBlock* b;
    const char* nm;
    int rcap;
  };
  BlkAlloc blks[5] = {{&pl->enc, "enc", R0cap}, {&pl->dec, "dec", Rdcap}, {&pl->z3b, "z3", Fcap}, {&pl->dz1b, "dz1", Fcap},
                      {&pl->clfb, "clf", LNcap}};
  std::vector<std::pair<C8Buf*, BufRec>> pend;
  for (auto& ba : blks) {
    ba.b->H.resize(ba.b->hidden.size());
    ba.b->dPre.resize(ba.b->hidden.size());
    for (size_t i = 0; i < ba.b->hidden.size(); ++i) {
      const int fcap = ba.b->hidden[i].rcap;
      pend.push_back({&ba.b->H[i], C8(std::string(ba.nm) + ".H" + std::to_string(i), ba.rcap, fcap)});
      pend.push_back({&ba.b->dPre[i], C8(std::string(ba.nm) + ".dPre" + std::to_string(i), ba.rcap, fcap)});
    }
  }
  // classifier hidden layers: DrVAE's operand u = [z1 | z2f - z1 | 1] and the fp32 gradient of u (VFAE: u is the z1
  // rows of Zdec, its gradient goes straight to DZ1)
  BufRec r_U{}, r_dU{};
  const bool own_u = pl->clf_nh > 0 && a->kind == DRVAE_KIND_DRVAE;
  if (own_u) {
    r_U = C8("clf.U", LNcap, round_up(pl->clf_in + 1, 16));
    r_dU = F32("clf.dU", (size_t)LNcap * pl->clf_in);
  }
  pl->arena_bytes = ab.total;
  cudaError_t err = cudaMalloc(&pl->arena, pl->arena_bytes);
  if (err != cudaSuccess) {
    delete pl;
    return set_cuda_error("drvae_plan_create: cudaMalloc(workspace)", err);
  }
  cudaMemset(pl->arena, 0, pl->arena_bytes);
  cudaMalloc(&pl->d_dyn, sizeof(StepDyn));
  cudaMemset(pl->d_dyn, 0, sizeof(StepDyn));
  if (const char* knob = getenv("DRVAE_B200_STEPK")) pl->stepk_enabled = atoi(knob) != 0;
  if (const char* knob = getenv("DRVAE_B200_DWA_EARLY_SMS")) pl->dwa_early_sms = std::max(0, atoi(knob));
  cudaMalloc(&pl->d_stepk_bar, 2 * sizeof(unsigned int));
  cudaMemset(pl->d_stepk_bar, 0, 2 * sizeof(unsigned int));
  {
    // the main chain outranks the side branch: when both have CTAs waiting for an SM (the side stream's wide row kernels
    // vs the next GEMM of the critical path) the critical path goes first
    int prio_least = 0, prio_greatest = 0;
    cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest);
    cudaStreamCreateWithPriority(&pl->s_main, cudaStreamNonBlocking, prio_greatest);
    cudaStreamCreateWithPriority(&pl->s_side, cudaStreamNonBlocking, prio_least);
    cudaStreamCreateWithPriority(&pl->s_dwa, cudaStreamNonBlocking, prio_least);
    for (int i = 0; i < drvae_plan::StepEvents::N; ++i) cudaEventCreateWithFlags(pl->ev.all() + i, cudaEventDisableTiming);
  }
  pl->bucket_ev.resize(pl->buckets.size());
  for (auto& ev : pl->bucket_ev) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
  cudaMalloc(&pl->dbg, sizeof(DebugWord));
  cudaMemset(pl->dbg, 0, sizeof(DebugWord));
  cudaMalloc(&pl->d_tabs, pl->h_tabs.size() * sizeof(int));
  cudaMemcpy(pl->d_tabs, pl->h_tabs.data(), pl->h_tabs.size() * sizeof(int), cudaMemcpyHostToDevice);
  if (!pl->wn_rows.empty()) {
    cudaMalloc(&pl->d_wn_rows, pl->wn_rows.size() * sizeof(WnRow));
    cudaMemcpy(pl->d_wn_rows, pl->wn_rows.data(), pl->wn_rows.size() * sizeof(WnRow), cudaMemcpyHostToDevice);
  }
  cudaMalloc(&pl->d_segs, pl->segs.size() * sizeof(Seg));
  cudaMemcpy(pl->d_segs, pl->segs.data(), pl->segs.size() * sizeof(Seg), cudaMemcpyHostToDevice);
  for (auto& pr : pend) *pr.first = c8_of(pl, pr.second);

  pl->shadow = mbuf_of<bf16>(pl, r_shadow);
  pl->derived = mbuf_of<float>(pl, r_derived);
  pl->eps_own = mbuf_of<float>(pl, r_eps);
  pl->dY5 = c8_of(pl, r_dY5);

  DevView& v = pl->view;
  memset(&v, 0, sizeof(v));
  v.kind = a->kind;
  v.X = X;
  v.Y = Y;
  v.Z = Z;
  v.Z3 = Z3;
  v.L = L;
  v.Ncap = Ncap;
  v.Xc = Xc;
  v.Zc = Zc;
  v.Z3c = Z3c;
  v.Zs = Zs;
  v.Z3s = Z3s;
  v.clf_ld = round_up(pl->clf_pin, 4);
  v.R0cap = R0cap;
  v.LNcap = LNcap;
  v.Rdcap = Rdcap;
  v.Fcap = Fcap;
  v.Flcap = Flcap;
  v.has_pair = pl->has_pair;
  v.has_T = pl->has_T;
  v.has_clf = pl->has_clf;
  v.has_fprop = pl->has_fprop;
  v.clf_in = pl->clf_in;
  v.counts = mbuf_of<int>(pl, r_counts);
  v.coefs = mbuf_of<float>(pl, r_coefs);
  v.pair_of = mbuf_of<int>(pl, r_pair_of);
  v.row_of_pair = mbuf_of<int>(pl, r_row_of_pair);
  v.ebase = mbuf_of<int>(pl, r_ebase);
  v.lab = mbuf_of<int>(pl, r_lab);
  v.ycls = mbuf_of<int>(pl, r_ycls);
  v.e_row = mbuf_of<int>(pl, r_e_row);
  v.e_jj = mbuf_of<int>(pl, r_e_jj);
  v.e_cls_full = mbuf_of<int>(pl, r_e_cls);
  v.tgt4 = mbuf_of<float4>(pl, r_tgt);
  v.Ain = c8_of(pl, r_Ain);
  v.Q = mbuf_of<float>(pl, r_Q);
  v.Z1f = mbuf_of<float>(pl, r_Z1f);
  v.Zdec = c8_of(pl, r_Zdec);
  v.Z1e = c8_of(pl, r_Z1e);
  v.PT = mbuf_of<float>(pl, r_PT);
  v.Z2Ff = mbuf_of<float>(pl, r_Z2Ff);
  v.QY = mbuf_of<float>(pl, r_QY);
  v.Q3 = mbuf_of<float>(pl, r_Q3);
  v.Z3b = c8_of(pl, r_Z3b);
  v.PZ1 = mbuf_of<float>(pl, r_PZ1);
  v.klq_row = mbuf_of<float>(pl, r_klq);
  v.klz2_row = mbuf_of<float>(pl, r_klz2);
  v.yl_row = mbuf_of<float>(pl, r_yl);
  v.ycat_row = mbuf_of<float>(pl, r_ycat);
  v.kfp_row = mbuf_of<float>(pl, r_kfp);
  v.kfpw_row = mbuf_of<float>(pl, r_kfpw);
  v.dec_part = mbuf_of<float>(pl, r_part);
  v.dec_tiles = dec_tiles;
  v.dY9 = c8_of(pl, r_dY9);
  v.dY7 = c8_of(pl, r_dY7);
  v.dYT = c8_of(pl, r_dYT);
  v.dY2 = c8_of(pl, r_dY2);
  v.dQ1e = mbuf_of<float>(pl, r_dQ1e);
  v.dQ2 = mbuf_of<float>(pl, r_dQ2);
  v.dZ3 = mbuf_of<float>(pl, r_dZ3);
  v.dZ1e = mbuf_of<float>(pl, r_dZ1e);
  v.dZdec = mbuf_of<float>(pl, r_dZdec);
  v.dZ1T = mbuf_of<float>(pl, r_dZ1T);
  v.DZ1 = mbuf_of<float>(pl, r_DZ1);
  v.DZ2F = mbuf_of<float>(pl, r_DZ2F);
  v.dlogit = mbuf_of<float>(pl, r_dlogit);
  v.clf_part = mbuf_of<float>(pl, r_clfp);
  v.loss_part = mbuf_of<float>(pl, r_lossp);
  v.losses = mbuf_of<float>(pl, r_losses);
  v.clf_w_off = pl->clf_w_off;
  v.clf_b_off = pl->clf_b_off;
  if (pl->clf_nh > 0) {
    ClfView& c = pl->clfv;
    c.nh = pl->clf_nh;
    c.pin = pl->clf_pin;
    c.U = own_u ? c8_of(pl, r_U) : v.Zdec;
    c.H = pl->clfb.H.back();
    c.D = pl->clfb.dPre.back();
    if (own_u) c.dU = mbuf_of<float>(pl, r_dU);
    cudaMalloc(&pl->d_clfv, sizeof(ClfView));
    cudaMemcpy(pl->d_clfv, &c, sizeof(ClfView), cudaMemcpyHostToDevice);
    v.clf = pl->d_clfv;
  }
  *out = pl;
  return 0;
}

extern "C" int drvae_plan_destroy(drvae_plan_t* pl) {
  if (!pl) return 0;
  drop_graphs(pl);
  if (pl->d_dyn) cudaFree(pl->d_dyn);
  if (pl->arena) cudaFree(pl->arena);
  if (pl->dbg) cudaFree(pl->dbg);
  if (pl->d_segs) cudaFree(pl->d_segs);
  if (pl->d_tabs) cudaFree(pl->d_tabs);
  if (pl->d_wn_rows) cudaFree(pl->d_wn_rows);
  if (pl->d_dwa_layers) cudaFree(pl->d_dwa_layers);
  if (pl->d_dwa_maps) cudaFree(pl->d_dwa_maps);
  if (pl->dp_counts) cudaFree(pl->dp_counts);
  if (pl->f32ws) cudaFree(pl->f32ws);
  if (pl->d_trace) cudaFree(pl->d_trace);
  if (pl->d_dwa_stats) cudaFree(pl->d_dwa_stats);
  if (pl->d_stepk_bar) cudaFree(pl->d_stepk_bar);
  if (pl->d_member_hp) cudaFree(pl->d_member_hp);
  if (pl->d_clfv) cudaFree(pl->d_clfv);
  if (pl->d_member) cudaFree(pl->d_member);
  if (pl->h_member_stage) cudaFreeHost(pl->h_member_stage);
  if (pl->member_ev) cudaEventDestroy(pl->member_ev);
  for (auto& ev : pl->bucket_ev) cudaEventDestroy(ev);
  for (int i = 0; i < drvae_plan::StepEvents::N; ++i)
    if (pl->ev.all()[i]) cudaEventDestroy(pl->ev.all()[i]);
  for (cudaStream_t s : {pl->s_main, pl->s_side, pl->s_dwa})
    if (s) cudaStreamDestroy(s);
  delete pl;
  return 0;
}

extern "C" long long drvae_plan_param_count(const drvae_plan_t* pl) { return pl ? pl->P : -1; }
extern "C" int drvae_plan_num_tensors(const drvae_plan_t* pl) { return pl ? (int)pl->tensors.size() : -1; }
extern "C" int drvae_plan_tensor_info(const drvae_plan_t* pl, int index, char* name, int name_cap, int* rows, int* cols,
                                      long long* offset) {
  if (!pl || index < 0 || index >= (int)pl->tensors.size()) return set_error("drvae_plan_tensor_info: bad index");
  const ParamInfo& t = pl->tensors[index];
  if (name && name_cap > 0) {
    strncpy(name, t.name.c_str(), name_cap - 1);
    name[name_cap - 1] = 0;
  }
  if (rows) *rows = t.rows;
  if (cols) *cols = t.cols;
  if (offset) *offset = t.off;
  return 0;
}
extern "C" int drvae_plan_tensor_ld(const drvae_plan_t* pl, int index) {
  if (!pl || index < 0 || index >= (int)pl->tensors.size()) return -1;
  return pl->tensors[index].ld;
}
extern "C" int drvae_plan_eps_layout(const drvae_plan_t* pl, drvae_eps_layout_t* out) {
  if (!pl || !out) return set_error("drvae_plan_eps_layout: null argument");
  *out = pl->epsl;
  return 0;
}
extern "C" long long drvae_plan_workspace_bytes(const drvae_plan_t* pl) { return pl ? (long long)pl->arena_bytes : -1; }
extern "C" int drvae_plan_num_buckets(const drvae_plan_t* pl) { return pl ? (int)pl->buckets.size() : -1; }
extern "C" int drvae_plan_bucket_info(const drvae_plan_t* pl, int index, long long* offset, long long* count) {
  if (!pl || index < 0 || index >= (int)pl->buckets.size()) return set_error("drvae_plan_bucket_info: bad index");
  if (offset) *offset = pl->buckets[index].first;
  if (count) *count = pl->buckets[index].second;
  return 0;
}
extern "C" int drvae_stream_wait_bucket(drvae_plan_t* pl, int index, void* stream) {
  if (!pl || index < 0 || index >= (int)pl->bucket_ev.size()) return set_error("drvae_stream_wait_bucket: bad index");
  cudaError_t err = cudaStreamWaitEvent((cudaStream_t)stream, pl->bucket_ev[index], 0);
  if (err != cudaSuccess) return set_cuda_error("drvae_stream_wait_bucket", err);
  return 0;
}
extern "C" long long drvae_plan_launch_count(const drvae_plan_t* pl) { return pl ? pl->launches : -1; }
extern "C" int drvae_set_gemm_impl(drvae_plan_t* pl, int impl) {
  if (!pl || (impl != GEMM_IMPL_TC && impl != GEMM_IMPL_SIMT)) return set_error("drvae_set_gemm_impl: bad argument");
  if (pl->gemm_impl != impl) drop_graphs(pl);  // captured sequences replay the kernels of the old implementation
  pl->gemm_impl = impl;
  return 0;
}
extern "C" int drvae_set_step_kernel(drvae_plan_t* pl, int enable) {
  if (!pl) return set_error("drvae_set_step_kernel: null plan");
  if (pl->stepk_enabled != (enable != 0)) drop_graphs(pl);
  pl->stepk_enabled = enable != 0;
  return 0;
}
extern "C" long long drvae_plan_step_kernel_launches(const drvae_plan_t* pl) { return pl ? pl->stepk_launches : -1; }
extern "C" int drvae_set_activation(drvae_plan_t* pl, int act) {
  if (!pl) return set_error("drvae_set_activation: null plan");
  if (act != DRVAE_ACT_ELU && act != DRVAE_ACT_SOFTPLUS)
    return set_error("drvae_set_activation: act must be DRVAE_ACT_ELU (0) or DRVAE_ACT_SOFTPLUS (1)");
  // captured sequences (and the step kernel's op tables inside them) launch the old activation's epilogue instances;
  // an uncaptured step records its tables afresh
  if (pl->act != act) drop_graphs(pl);
  pl->act = act;
  return 0;
}
extern "C" int drvae_debug_side_delay(drvae_plan_t* pl, long long cycles) {
  if (!pl || cycles < 0) return set_error("drvae_debug_side_delay: bad argument");
  pl->side_delay_cycles = cycles;
  drop_graphs(pl);
  return 0;
}

namespace {

// Layer table + tensor maps of the grouped dW+Adam launch.  Leaves pl->dwa_ok false (-> train steps run gradient +
// stand-alone Adam) when the optimizer state is not bound, with weight norm (the update acts on (v, g)), with more
// than DWA_MAX_LAYERS layers, or when a layer does not meet the kernel's layout conditions (class columns must share
// the 128-feature tile of the ones column).
int build_dwa(drvae_plan* pl) {
  pl->dwa_ok = false;
  pl->dwa_layers.clear();
  if (!pl->params || !pl->adam_m || !pl->adam_v || pl->wn) return 0;
  struct Ref {
    const Shadow* W;
    const C8Buf* dY;
    const C8Buf* X;
    int cnt, skip;
  };
  std::vector<Ref> refs;
  const DevView& v = pl->view;
  auto add_block = [&](MlpBlock& b, const C8Buf* dYh, const C8Buf* in, int cnt) {
    const int n = (int)b.hidden.size();
    refs.push_back({&b.head, dYh, &b.H[n - 1], cnt, -1});
    for (int i = 0; i < n; ++i) refs.push_back({&b.hidden[i], &b.dPre[i], i == 0 ? in : &b.H[i - 1], cnt, -1});
  };
  add_block(pl->dec, &pl->dY5, &v.Zdec, CNT_RD);
  add_block(pl->enc, &v.dY2, &v.Ain, CNT_R0);
  if (pl->has_fprop) {
    add_block(pl->z3b, &v.dY7, &v.Z1e, CNT_F);
    add_block(pl->dz1b, &v.dY9, &v.Z3b, CNT_F);
  }
  if (pl->has_T) refs.push_back({&pl->Tsh, &v.dYT, &v.Zdec, CNT_LN, pl->arch.kind == DRVAE_KIND_PVAE ? CNT_NP : -1});
  for (int i = 0; i < pl->clf_nh; ++i)
    refs.push_back({&pl->clfb.hidden[i], &pl->clfb.dPre[i], i == 0 ? &pl->clfv.U : &pl->clfb.H[i - 1], CNT_LN, -1});
  if ((int)refs.size() > DWA_MAX_LAYERS) return 0;
  // heaviest layers first: the strided persistent grid then ends on the small ones
  std::stable_sort(refs.begin(), refs.end(), [](const Ref& a, const Ref& b) {
    return (long long)a.W->kc * a.W->rcap > (long long)b.W->kc * b.W->rcap;
  });
  std::vector<DwaMaps> maps(refs.size());
  int tile = 0;
  for (size_t i = 0; i < refs.size(); ++i) {
    const Shadow& W = *refs[i].W;
    const int cc = W.kaug - W.kin - 1;
    if (cc > 0 && (W.kin % GEMM_BM) + 1 + cc > GEMM_BM) return 0;
    if (W.BN % DWA_R || W.BN > 256 || W.rcap != W.BN * W.tiles_n || W.ntens > 2 || (W.ld & 3)) return 0;
    if (W.ntens == 2 && (W.ilv_block % DWA_R)) return 0;
    DwaLayer y{};
    y.tile_begin = tile;
    y.tiles_m = cdiv(W.kaug, GEMM_BM);
    y.tiles_n = W.tiles_n;
    y.BN = W.BN;
    tile += y.tiles_m * y.tiles_n * pl->E;
    y.tile_end = tile;
    y.kin = W.kin;
    y.kaug = W.kaug;
    y.cnt_which = refs[i].cnt;
    y.a_row0 = 0;
    y.ntens = W.ntens;
    y.rows_each = W.rows_each[0];
    y.ilv_block = W.ilv_block;
    y.ilv_stride = W.ilv_stride;
    y.rcap = W.rcap;
    y.skip_which = refs[i].skip;
    y.tab_off = W.tab_off;
    y.drv_bias_off = W.bias_off;
    y.drv_clsb_off = W.clsb_off;
    y.drv_clsb_ld = W.rcap;
    y.ld = W.ld;
    y.w_off[0] = W.w_off[0];
    y.w_off[1] = W.ntens > 1 ? W.w_off[1] : W.w_off[0];
    y.sh_off = W.off;
    pl->dwa_layers.push_back(y);
    DwaMaps& m = maps[i];
    const C8Buf& X = *refs[i].X;
    const C8Buf& dY = *refs[i].dY;
    cudaError_t err = gemm_c8_map(&m.A, GemmOperand{X.p, X.ms, X.rcap, X.fcap >> 3, 0}, pl->E, GEMM_BK, GEMM_BM / 8);
    if (err == cudaSuccess) err = gemm_c8_map(&m.B, GemmOperand{dY.p, dY.ms, dY.rcap, dY.fcap >> 3, 0}, pl->E, GEMM_BK, W.BN / 8);
    if (err == cudaSuccess)
      err = gemm_c8_map(&m.S, GemmOperand{pl->shadow.p + W.off, pl->shadow.ms, W.rcap, W.kc >> 3, 0}, pl->E, DWA_R, GEMM_BM / 8);
    for (int w = 0; w < 2 && err == cudaSuccess; ++w) {
      const int ww = w < W.ntens ? w : 0;
      err = dwa_state_map(&m.P[w], pl->params + W.w_off[ww], W.ld, W.rows_each[ww], pl->P, pl->E);
      if (err == cudaSuccess) err = dwa_state_map(&m.M[w], pl->adam_m + W.w_off[ww], W.ld, W.rows_each[ww], pl->P, pl->E);
      if (err == cudaSuccess) err = dwa_state_map(&m.V[w], pl->adam_v + W.w_off[ww], W.ld, W.rows_each[ww], pl->P, pl->E);
    }
    if (err != cudaSuccess) return set_cuda_error("drvae_plan_bind: tensor maps of the grouped weight-gradient launch", err);
  }
  if (!pl->d_dwa_layers) cudaMalloc(&pl->d_dwa_layers, sizeof(DwaLayer) * DWA_MAX_LAYERS);
  if (!pl->d_dwa_maps) cudaMalloc(&pl->d_dwa_maps, sizeof(DwaMaps) * DWA_MAX_LAYERS);
  cudaError_t err = cudaMemcpy(pl->d_dwa_layers, pl->dwa_layers.data(), sizeof(DwaLayer) * pl->dwa_layers.size(), cudaMemcpyHostToDevice);
  if (err == cudaSuccess) err = cudaMemcpy(pl->d_dwa_maps, maps.data(), sizeof(DwaMaps) * maps.size(), cudaMemcpyHostToDevice);
  if (err != cudaSuccess) return set_cuda_error("drvae_plan_bind: uploading the grouped weight-gradient tables", err);
  pl->dwa_tiles = tile;
  pl->dwa_early_tiles = (!refs.empty() && refs[0].W == &pl->dec.head) ? pl->dwa_layers[0].tile_end : 0;
  pl->dwa_ok = true;
  return 0;
}

}  // namespace

extern "C" int drvae_plan_bind(drvae_plan_t* pl, float* params, float* adam_m, float* adam_v, float* grads) {
  if (!pl || !params) return set_error("drvae_plan_bind: params must not be null");
  pl->params = params;
  pl->adam_m = adam_m;
  pl->adam_v = adam_v;
  pl->grads = grads;
  pl->shadows_valid = false;
  drop_graphs(pl);  // captured sequences hold the old pointers
  return build_dwa(pl);
}

extern "C" int drvae_debug_buffer(drvae_plan_t* pl, const char* name, void** ptr, long long* ms_bytes, long long* bytes,
                                  int* rcap, int* fcap) {
  if (!pl || !name) return set_error("drvae_debug_buffer: null argument");
  auto it = pl->bufs.find(name);
  if (it == pl->bufs.end()) return set_error("drvae_debug_buffer: unknown buffer");
  if (ptr) *ptr = pl->arena + it->second.off;
  if (ms_bytes) *ms_bytes = (long long)it->second.ms_bytes;
  if (bytes) *bytes = (long long)it->second.bytes;
  if (rcap) *rcap = it->second.rcap;
  if (fcap) *fcap = it->second.fcap;
  return 0;
}

// =============================================================================================
// step executor
// =============================================================================================
namespace {

void prof_pre(drvae_plan* pl, cudaStream_t st, const std::string& tag) {
  if (!pl->prof_on) return;
  if (pl->prof_used + 2 > pl->prof_ev.size()) {
    for (int i = 0; i < 256; ++i) {
      cudaEvent_t e;
      cudaEventCreate(&e);
      pl->prof_ev.push_back(e);
    }
  }
  pl->prof_tags.push_back(tag);
  cudaEventRecord(pl->prof_ev[pl->prof_used++], st);
}
void prof_post(drvae_plan* pl, cudaStream_t st) {
  if (!pl->prof_on) return;
  cudaEventRecord(pl->prof_ev[pl->prof_used++], st);
}

// Where the readers of per-member scalars look (MemberScalars in plan.h): the shared copy in the per-step block with
// stride 0, or the member table's per-step expansion.
const MemberScalars* member_base(const drvae_plan* pl) { return pl->member_table ? pl->d_member : &pl->d_dyn->s.mem; }
const AdamHyper* member_adam(const drvae_plan* pl) { return &member_base(pl)->adam; }
int member_adam_ms(const drvae_plan* pl) { return pl->member_table ? (int)sizeof(MemberScalars) : 0; }
MemberExpand member_expand(const drvae_plan* pl) {
  return pl->member_table ? MemberExpand{pl->d_member_hp, pl->d_member, pl->E} : MemberExpand{nullptr, nullptr, 0};
}
int set_dyn_threads(const MemberExpand& mx) { return mx.n > 0 ? std::min(256, (mx.n + 31) / 32 * 32) : 1; }

struct Exec {
  drvae_plan* pl;
  cudaStream_t st;
  DevView v;
  int N;
  cudaError_t err = cudaSuccess;
  const char* phase = "";
  std::string sub = "head";  // layer within the current block: h0, h1, ..., head
  bool splitk = false;       // split-K weight gradients (large minibatches, gradient path)
  bool defer_dw = false;     // fused train step: weight gradients + Adam of every layer in ONE launch at the end of
                             // backward (dwadam.cuh) instead of the per-layer gradient GEMMs
  StepRecorder* rec = nullptr;  // non-null: launches are recorded as ops of the persistent step kernel (stepk.cuh)
  // stand-alone weight-gradient GEMMs (gradient path: they feed nothing but the optimizer / the gradient exchange) leave
  // the dX chain for this stream; each waits for what has been enqueued on the chain's stream so far (its dY and input)
  cudaStream_t dw_stream = nullptr;
  cudaEvent_t dw_event = nullptr;
  int cta_cap = 0;                          // > 0: persistent GEMM grids are capped (SMs reserved for the early dW+Adam launch)
  std::function<void()> after_head_dx;      // called once after the next block_bwd has enqueued its head dX GEMM
  bool ok() const { return err == cudaSuccess; }
  // stream dependencies: real events, or level bookkeeping while recording
  void ev_record(cudaEvent_t ev, cudaStream_t s) {
    if (rec)
      rec->record_event(ev, s);
    else
      cudaEventRecord(ev, s);
  }
  void ev_wait(cudaStream_t s, cudaEvent_t ev) {
    if (rec)
      rec->wait_event(s, ev);
    else
      cudaStreamWaitEvent(s, ev, 0);
  }
  // one row operation: `per_model` items of STEPK_ROWS rows (or kernel-specific blocks) per ensemble member
  template <class F>
  void row_op(int kind, const char* name, int per_model, int arg, F&& real_launch) {
    if (!ok()) return;
    if (rec) {
      rec->add_row(kind, per_model, pl->E, arg, st, std::string(phase) + ":" + name);
      return;
    }
    pre(name);
    real_launch();
    chk();
  }
  // event bracket around one launch when profiling is on
  void pre(const std::string& op) {
    prof_pre(pl, st, std::string(phase) + ":" + op);
    v.trace = nullptr;
    if (pl->trace_on && pl->trace_next < pl->trace_cap) {
      v.trace = pl->d_trace;
      v.trace_id = pl->trace_next++;
      pl->trace_tags.push_back(std::string(phase) + ":" + op);
    }
  }
  void post() { prof_post(pl, st); }
  void chk() {
    post();
    if (err == cudaSuccess) err = cudaGetLastError();
    pl->launches++;
  }

  const int* cnt(int which) const { return v.counts.p + which; }

  GemmOperand op_c8(const C8Buf& b, int row0) const { return GemmOperand{b.p, b.ms, b.rcap, b.fcap >> 3, row0}; }
  GemmOperand op_shadow(const Shadow& s) const {
    return GemmOperand{pl->shadow.p + s.off, pl->shadow.ms, s.rcap, s.kc >> 3, 0};
  }
  EpiParams epi_base() const {
    EpiParams e;
    memset(&e, 0, sizeof(e));
    return e;
  }
  void launch(int epi, GemmProblem& p, const EpiParams& e, const char* op) {
    if (!ok()) return;
    p.dbg = pl->dbg;
    p.desc_variant = 0;
    if (p.ksplit < 1) p.ksplit = 1;
    p.ens = pl->E;
    p.max_ctas = cta_cap;
    if (rec) {
      p.trace = nullptr;
      p.trace_id = 0;
      rec->add_gemm(epi, p, e, pl->E, st, std::string(phase) + ":" + op);
      return;
    }
    pre(op);
    p.trace = v.trace;
    p.trace_id = v.trace_id;
    cudaError_t r = gemm_launch(epi, p, e, pl->E, pl->gemm_impl, st);
    post();
    if (r != cudaSuccess) err = r;
    pl->launches++;
  }

  // D[rows, W.rcap] = A[rows, kin] . W^T
  void gemm_nt(const C8Buf& A, int a_row0, const Shadow& W, int epi, EpiParams e, int dyn_which, int row_bound) {
    GemmProblem p{};
    p.A = op_c8(A, a_row0);
    p.B = op_shadow(W);
    p.mode = GEMM_NT;
    p.M = row_bound;
    p.N = W.rcap;
    p.K = W.kc;
    p.dyn = cnt(dyn_which);
    p.dyn_stride = (int)v.counts.ms;
    p.BN = W.BN;
    p.tiles_n = W.tiles_n;
    p.tiles_m = cdiv(row_bound, GEMM_BM);
    launch(epi, p, e, (std::string(epi == EPI_DECLOSS ? "gemm_nt_decloss." : "gemm_nt.") + sub).c_str());
  }
  // D[rows, kin] = dY[rows, nout] . W
  void gemm_dx(const C8Buf& dY, const Shadow& W, int epi, EpiParams e, int dyn_which, int row_bound) {
    GemmProblem p{};
    p.A = op_c8(dY, 0);
    p.B = op_shadow(W);
    p.mode = GEMM_DX;
    p.M = row_bound;
    p.N = W.kc;
    p.K = round_up(W.nout_total, 16);
    p.dyn = cnt(dyn_which);
    p.dyn_stride = (int)v.counts.ms;
    p.BN = W.BNx;
    p.tiles_n = W.tiles_nx;
    p.tiles_m = cdiv(row_bound, GEMM_BM);
    launch(epi, p, e, ("gemm_dx." + sub).c_str());
  }
  // grad W^T[kaug, nout] = Xin[rows, kaug]^T . dY[rows, nout]: weight, bias (ones column) and class-column
  // gradients of one layer into the gradient buffer.
  void gemm_dw(const C8Buf& dY, const C8Buf& Xin, int x_row0, const Shadow& W, int dyn_which, int row_bound) {
    if (defer_dw) return;
    GemmProblem p{};
    p.A = op_c8(Xin, x_row0);
    p.B = op_c8(dY, 0);
    p.mode = GEMM_DW;
    p.M = W.kaug;
    p.N = W.rcap;
    p.K = row_bound;
    p.dyn = cnt(dyn_which);
    p.dyn_stride = (int)v.counts.ms;
    p.BN = W.BN;
    p.tiles_n = W.tiles_n;
    p.tiles_m = cdiv(W.kaug, GEMM_BM);
    p.ksplit = 1;
    if (splitk) {
      // large minibatch, few weight tiles: split the contraction (rows) so the persistent grid is filled;
      // partial tiles accumulate with red.global.add into the gradient buffer zeroed at the start of the step
      const int nkb = cdiv(row_bound, GEMM_BK);
      const int tiles = p.tiles_m * p.tiles_n * pl->E;
      int ks = std::min(cdiv(2 * gemm_num_sms(), tiles), nkb / 4);
      p.ksplit = std::max(1, std::min(ks, 64));
    }
    EpiParams e = epi_base();
    e.grad = v.grads.p;
    e.grad_ms = v.grads.ms;
    e.g_tab = pl->d_tabs + W.tab_off;
    e.g_tab_n = W.rcap;
    e.g_kin = W.kin;
    e.g_kaug = W.kaug;
    const bool aside = dw_stream && dw_stream != st;
    cudaStream_t chain_st = st;
    if (aside) {
      if (rec) {
        rec->after(dw_stream, st);
      } else {
        cudaEventRecord(dw_event, st);
        cudaStreamWaitEvent(dw_stream, dw_event, 0);
      }
      st = dw_stream;
    }
    launch(EPI_GRAD, p, e, ("gemm_dw." + sub).c_str());
    st = chain_st;
  }

  // the hidden-layer activation's forward (bias + activation -> bf16 chunk8) and backward (* activation') epilogues
  int act_fwd_epi() const { return pl->act == DRVAE_ACT_SOFTPLUS ? EPI_SP_C8 : EPI_ELU_C8; }
  int act_bwd_epi() const { return pl->act == DRVAE_ACT_SOFTPLUS ? EPI_DSP_C8 : EPI_DACT_C8; }
  EpiParams epi_act(const Shadow& W, const C8Buf& out, int width, bool class_aug) const {
    EpiParams e = epi_base();
    e.out_c8 = out.p;
    e.out_c8_ms = out.ms;
    e.out_c8_rcap = out.rcap;
    e.n_valid = width;
    e.bias = pl->derived.p + W.bias_off;
    e.bias_ms = pl->derived.ms;
    if (class_aug) {
      e.clsb = pl->derived.p + W.clsb_off;
      e.clsb_ms = pl->derived.ms;
      e.clsb_ld = W.rcap;
      e.row_cls = v.e_cls_full.p;
      e.row_cls_ms = v.e_cls_full.ms;
    }
    return e;
  }
  EpiParams epi_f32(float* out, long long ms, int ld, int n_valid, const Shadow* bias_of) const {
    EpiParams e = epi_base();
    e.out_f32 = out;
    e.out_f32_ms = ms;
    e.out_ld = ld;
    e.n_valid = n_valid;
    if (bias_of) {
      e.bias = pl->derived.p + bias_of->bias_off;
      e.bias_ms = pl->derived.ms;
    }
    return e;
  }
  EpiParams epi_dact(const C8Buf& act, const C8Buf& out, int width) const {
    EpiParams e = epi_base();
    e.out_c8 = out.p;
    e.out_c8_ms = out.ms;
    e.out_c8_rcap = out.rcap;
    e.act = act.p;
    e.act_ms = act.ms;
    e.act_rcap = act.rcap;
    e.n_valid = width;
    return e;
  }

  // hidden layers of a block: in -> H[0] -> ... -> H[n-1]
  void block_hidden_fwd(MlpBlock& b, const C8Buf& in, int in_row0, int dyn_which, int row_bound) {
    for (size_t i = 0; i < b.hidden.size(); ++i) {
      const C8Buf& src = (i == 0) ? in : b.H[i - 1];
      sub = "h" + std::to_string(i);
      gemm_nt(src, i == 0 ? in_row0 : 0, b.hidden[i], act_fwd_epi(), epi_act(b.hidden[i], b.H[i], b.widths[i], b.class_aug && i == 0),
              dyn_which, row_bound);
    }
    sub = "head";
  }
  // backward of a block given the head gradient rows dYh; optionally the input gradient as fp32.
  // Per layer the input gradient (the next layer's input, on the critical path) is launched before the
  // weight gradient (which feeds nothing but the optimizer).
  void block_bwd(MlpBlock& b, const C8Buf& dYh, const C8Buf& in, int in_row0, int in_feat, float* dx_out, long long dx_ms,
                 int dyn_which, int row_bound) {
    const int n = (int)b.hidden.size();
    sub = "head";
    gemm_dx(dYh, b.head, act_bwd_epi(), epi_dact(b.H[n - 1], b.dPre[n - 1], b.widths[n - 1]), dyn_which, row_bound);
    if (after_head_dx) {
      auto hook = std::move(after_head_dx);
      after_head_dx = nullptr;
      hook();
    }
    gemm_dw(dYh, b.H[n - 1], 0, b.head, dyn_which, row_bound);
    block_bwd_hidden(b, in, in_row0, in_feat, dx_out, dx_ms, dyn_which, row_bound);
  }
  // backward of the hidden layers given dPre of the last one (written by the head's dX GEMM, or by a row kernel for a
  // block without a GEMM head: the classifier)
  void block_bwd_hidden(MlpBlock& b, const C8Buf& in, int in_row0, int in_feat, float* dx_out, long long dx_ms, int dyn_which,
                        int row_bound) {
    const int n = (int)b.hidden.size();
    for (int i = n - 1; i >= 0; --i) {
      const C8Buf& src = (i == 0) ? in : b.H[i - 1];
      sub = "h" + std::to_string(i);
      if (i > 0) {
        gemm_dx(b.dPre[i], b.hidden[i], act_bwd_epi(), epi_dact(b.H[i - 1], b.dPre[i - 1], b.widths[i - 1]), dyn_which, row_bound);
      } else if (dx_out) {
        gemm_dx(b.dPre[0], b.hidden[0], EPI_STORE_F32, epi_f32(dx_out, dx_ms, in_feat, in_feat, nullptr), dyn_which, row_bound);
      }
      gemm_dw(b.dPre[i], src, i == 0 ? in_row0 : 0, b.hidden[i], dyn_which, row_bound);
    }
    sub = "head";
  }
};

// Step-dependent Adam scalars, computed once on the host so that the grouped dW+Adam launch and the
// stand-alone kernel apply bit-identical updates.  bc1_out: the bias correction lr is divided by (member tables).
AdamHyper adam_scalars(const drvae_hparams_t* hp, float* bc1_out) {
  const double t = (double)hp->step + 1.0;
  const float bc1 = (float)(1.0 - pow((double)hp->beta1, t));
  const float bc2 = (float)(1.0 - pow((double)hp->beta2, t));
  *bc1_out = bc1;
  AdamHyper a;
  a.lr_bc1 = hp->lr / bc1;
  a.inv_sqrt_bc2 = 1.0f / sqrtf(bc2);
  a.beta1 = hp->beta1;
  a.beta2 = hp->beta2;
  a.eps = hp->adam_eps;
  a.wd = hp->weight_decay;
  return a;
}

int fill_view(drvae_plan* pl, Exec& ex, const drvae_batch_t* b, const drvae_noise_t* nz, const drvae_hparams_t* hp,
              bool need_grad) {
  if (!pl->params) return set_error("drvae: plan has no bound parameters (drvae_plan_bind)");
  if (!b || !b->x1) return set_error("drvae: batch.x1 is null");
  if (b->N < 1 || b->N > pl->Ncap) return set_error("drvae: batch.N exceeds the plan's max_batch");
  if (pl->has_pair && (!b->x2 || !b->has_x2)) return set_error("drvae: this model needs x2 and has_x2");
  if (pl->has_clf && (!b->y || !b->has_y)) return set_error("drvae: this model needs y and has_y");
  if (need_grad && !ex.defer_dw && !pl->grads) return set_error("drvae: no gradient buffer bound");
  DevView& v = ex.v;
  v = pl->view;
  const int N = b->N;
  ex.N = N;
  v.N = N;
  v.need_grad = need_grad;
  if (b->row_index && b->dataset_rows < 1) return set_error("drvae: batch.row_index needs dataset_rows >= 1");
  const long long drows = b->row_index ? b->dataset_rows : N;  // rows per model in the caller's arrays
  const long long rowsX = drows * pl->X;
  v.x1 = MBuf<const float>{b->x1, rowsX};
  v.x2 = MBuf<const float>{b->x2, rowsX};
  v.y = MBuf<const int>{b->y, drows};
  v.has_x2 = MBuf<const int>{b->has_x2, drows};
  v.has_y = MBuf<const int>{b->has_y, drows};
  v.row_index = MBuf<const int>{b->row_index, N};
  const float* eps = (nz && nz->eps) ? nz->eps : pl->eps_own.p;
  const long long ems = (nz && nz->eps) ? pl->epsl.total : pl->eps_own.ms;
  v.eps_x1 = MBuf<const float>{eps + pl->epsl.off_x1, ems};
  v.eps_x2 = MBuf<const float>{eps + pl->epsl.off_x2, ems};
  v.eps_z1 = MBuf<const float>{eps + pl->epsl.off_z1, ems};
  v.eps_z2 = MBuf<const float>{eps + pl->epsl.off_z2, ems};
  v.eps_z2f = MBuf<const float>{eps + pl->epsl.off_z2f, ems};
  v.eps_z3 = MBuf<const float>{eps + pl->epsl.off_z3, ems};
  v.own_noise = (nz && nz->eps) ? 0 : 1;
  v.dyn = pl->d_dyn;
  v.mem = member_base(pl);
  v.mem_stride = pl->member_table ? 1 : 0;
  v.params = MBuf<float>{pl->params, pl->P};
  v.clf_w = pl->wn ? MBuf<const float>{pl->derived.p + pl->clf_eff_off, pl->derived.ms}
                   : MBuf<const float>{pl->params + pl->clf_w_off, pl->P};
  v.grads = MBuf<float>{pl->grads, pl->P};
  v.adam_m = MBuf<float>{pl->adam_m, pl->P};
  v.adam_v = MBuf<float>{pl->adam_v, pl->P};
  return 0;
}

// per-step scalars of one call (written to device memory by set_dyn_kernel)
StepDyn make_dyn(const drvae_noise_t* nz, const drvae_hparams_t* hp, bool fused_adam) {
  StepDyn d{};
  StepScalars& s = d.s;
  s.kl_min = hp->kl_min;
  s.mem.noise_std = hp->noise_std;
  s.beta_pert = hp->beta_pert;
  s.mem.pertloss_rate = hp->pertloss_rate;
  s.mem.kl_qz2pz2_rate = hp->kl_qz2pz2_rate;
  s.mem.yloss_rate = hp->yloss_rate;
  s.training = hp->training;
  s.add_noise = hp->add_noise;
  s.gN = hp->global_N;
  s.gNp = hp->global_Np;
  s.gNlab = hp->global_Nlab;
  for (int j = 0; j < 8; ++j) s.mem.log_prior[j] = hp->log_prior_y[j];
  s.mem.adam = adam_scalars(hp, &d.bc1);
  s.fused_adam = fused_adam ? 1 : 0;
  d.noise_step = (unsigned)hp->step;
  d.noise_seed = nz ? nz->seed : 0ULL;
  d.row_offset = nz ? nz->row_offset : 0LL;
  d.counts_dev = hp->global_counts_dev;
  return d;
}

int push_dyn(drvae_plan* pl, const StepDyn& d, cudaStream_t st) {
  prof_pre(pl, st, ":set_dyn");
  const MemberExpand mx = member_expand(pl);
  launch_k(set_dyn_kernel, dim3(1), dim3(set_dyn_threads(mx)), 0, st, d, pl->d_dyn, mx);
  prof_post(pl, st);
  pl->launches++;
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) return set_cuda_error("set_dyn_kernel", err);
  return 0;
}

int run_adam(drvae_plan* pl, const drvae_hparams_t* hp, int update, cudaStream_t st) {
  if (!pl->params) return set_error("drvae: plan has no bound parameters");
  if (update && (!pl->adam_m || !pl->adam_v || !pl->grads)) return set_error("drvae: Adam needs bound moments and gradients");
  AdamArgs a{};
  a.params = MBuf<float>{pl->params, pl->P};
  a.grads = MBuf<float>{pl->grads, pl->P};
  a.m = MBuf<float>{pl->adam_m, pl->P};
  a.v = MBuf<float>{pl->adam_v, pl->P};
  a.shadow = pl->shadow;
  a.derived = pl->derived;
  a.segs = pl->d_segs;
  a.nseg = (int)pl->segs.size();
  a.P = pl->P;
  a.update = update;
  a.h = member_adam(pl);  // the caller has pushed this step's scalars
  a.h_ms = member_adam_ms(pl);
  // PVAE: p(z2|z1) takes part in the loss only through pair rows (PVAE.py:313-330); without pairs the reference's
  // gradient is None and torch.optim.Adam leaves the tensors (and their moments) untouched
  a.skip_lo = a.skip_hi = 0;
  if (pl->arch.kind == DRVAE_KIND_PVAE && pl->has_T) a.skip_lo = (int)pl->T_range[0], a.skip_hi = (int)(pl->T_range[0] + pl->T_range[1]);
  a.dyn = pl->d_dyn;
  a.counts = pl->view.counts.p;
  a.counts_stride = (int)pl->view.counts.ms;
  dim3 grid(cdiv(pl->P, 1024), pl->E);
  prof_pre(pl, st, update ? "opt:adam" : "opt:shadow_sync");
  adam_kernel<<<grid, 256, 0, st>>>(a);
  prof_post(pl, st);
  pl->launches++;
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) return set_cuda_error("adam_kernel", err);
  if (pl->wn) {
    // weight-normalised layers: the kernel-facing copies hold g v / ||v||, rebuilt row-wise
    WnArgs w{pl->d_wn_rows, (int)pl->wn_rows.size(), a.params, a.grads, pl->shadow, pl->derived};
    prof_pre(pl, st, "opt:wn_refresh");
    wn_refresh_kernel<<<dim3(cdiv(w.nrows, 8), pl->E), 256, 0, st>>>(w);
    prof_post(pl, st);
    pl->launches++;
    err = cudaGetLastError();
    if (err != cudaSuccess) return set_cuda_error("wn_refresh_kernel", err);
  }
  pl->shadows_valid = true;
  return 0;
}

// weight norm: effective-weight gradients -> (dv, dg), in place in the gradient buffer
int run_wn_grad(drvae_plan* pl, cudaStream_t st) {
  if (!pl->wn) return 0;
  WnArgs w{pl->d_wn_rows, (int)pl->wn_rows.size(), MBuf<float>{pl->params, pl->P}, MBuf<float>{pl->grads, pl->P}, pl->shadow,
           pl->derived};
  prof_pre(pl, st, "opt:wn_grad");
  wn_grad_kernel<<<dim3(cdiv(w.nrows, 8), pl->E), 256, 0, st>>>(w);
  prof_post(pl, st);
  pl->launches++;
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) return set_cuda_error("wn_grad_kernel", err);
  return 0;
}

// forward (+ optional backward) of one minibatch per model
//
// Schedule.  One launch sequence covers every member of the ensemble.  The main chain (encoder, p(z2|z1), decoder and
// the dX GEMMs back to the encoder) runs on the plan's high-priority stream: it forks from the caller's stream after
// the per-step scalars and joins it again before the grouped dW+Adam launch.  What is off that chain runs on the
// low-priority side stream: the latent-noise generator (next to the encoder GEMMs), the label-dependent branch
// (forward and backward) and the loss reduction.  The classifier weight gradient runs on the caller's stream, idle
// until the join, and the early part of the dW+Adam launch on a low-priority stream of its own.  Captured into a CUDA
// graph the forks and joins become graph edges.  The main chain stays on the caller's stream under per-launch
// profiling, under the step kernel and on the gradient path, whose bucket events the caller waits for on that stream
// (the stand-alone weight-gradient GEMMs then take the plan's main stream); profiling and plans without the
// label-dependent branch run on one stream.
int run_step(drvae_plan* pl, const drvae_batch_t* b, const drvae_noise_t* nz, const drvae_hparams_t* hp, float* losses_out,
             cudaStream_t st, bool backward, bool fused_adam) {
  if (!hp) return set_error("drvae: hparams is null");
  // (train_is_fused chooses the fused step only when the grouped launch is built, i.e. the moments are bound)
  if (fused_adam && !pl->dwa_ok) return set_error("drvae: the fused train step needs the grouped dW+Adam launch");
  Exec ex;
  ex.pl = pl;
  ex.st = st;
  ex.defer_dw = backward && fused_adam;
  int rc = fill_view(pl, ex, b, nz, hp, backward);
  if (rc) return rc;
  if (!pl->shadows_valid) {
    rc = run_adam(pl, hp, 0, st);
    if (rc) return rc;
  }
  DevView& v = ex.v;
  const int E = pl->E, N = ex.N, L = pl->L;
  const int R0b = (pl->has_pair ? 2 : 1) * N, LNb = L * N, Rdb = (pl->has_pair ? 3 : 1) * L * N;
  // row parallelism of the fixed-order reductions: sized for one wave at ensemble scale, widened for a single
  // model on a large minibatch
  // (functions of the row counts only, so an ensemble member sums in the same order as a single-model plan)
  v.clf_splits = std::max(CLF_SPLITS, std::min(CLF_SPLITS_MAX, cdiv(LNb, 64)));
  v.loss_slices = std::max(1, std::min(LOSS_SLICES_MAX, cdiv(Rdb, 512)));
  ex.splitk = backward && !fused_adam && Rdb >= 2048;
  if (ex.splitk) {
    cudaError_t e0 = cudaMemsetAsync(pl->grads, 0, sizeof(float) * (size_t)pl->P * E, st);
    if (e0 != cudaSuccess) return set_cuda_error("drvae: zeroing the gradient buffer", e0);
  }
  const int Fb = std::max(1, L * pl->Y * N);
  const bool own_eps = !(nz && nz->eps);
  if (own_eps) {
    long long most = 0;
    for (int inner : {pl->Z, pl->Y * pl->Z3}) most = std::max(most, (long long)L * N * ((inner + 3) / 4));
    if (most >= (1LL << 31)) return set_error("drvae: minibatch too large for the noise generator");
  }

  // Persistent step kernel (stepk.cuh): everything between the input preparation and the grouped dW+Adam launch is
  // recorded (same code below, same dependencies) and runs as ONE cooperative launch.
  const bool use_stepk = pl->stepk_enabled && !pl->stepk_unsupported && pl->gemm_impl == GEMM_IMPL_TC &&
                         pl->d_stepk_bar != nullptr;
  StepRecorder recorder;

  // the main chain on the plan's high-priority stream (see above)
  const bool own_main = !use_stepk && !pl->prof_on && !(backward && !fused_adam) && pl->has_fprop;
  if (own_main) cudaEventRecord(pl->ev.begin, st);

  // grouped weight-gradient + Adam launch over the tiles [t0, t1) (dwadam.cuh)
  auto launch_dwadam = [&](int t0, int t1, cudaStream_t stream, int max_ctas, const char* tag) {
    DwaParams dp{};
    dp.n_layers = (int)pl->dwa_layers.size();
    dp.n_models = E;
    dp.total_tiles = pl->dwa_tiles;
    dp.tile_begin = t0;
    dp.tile_end = t1;
    dp.layers = pl->d_dwa_layers;
    dp.maps = pl->d_dwa_maps;
    dp.tabs = pl->d_tabs;
    dp.counts = v.counts.p;
    dp.counts_stride = (int)v.counts.ms;
    dp.adam_p = pl->params;
    dp.adam_m = pl->adam_m;
    dp.adam_v = pl->adam_v;
    dp.state_ms = pl->P;
    dp.drv = pl->derived.p;
    dp.drv_ms = pl->derived.ms;
    dp.shadow = pl->shadow.p;
    dp.shadow_ms = pl->shadow.ms;
    dp.adam = member_adam(pl);
    dp.adam_ms = member_adam_ms(pl);
    dp.dbg = pl->dbg;
    cudaStream_t keep = ex.st;
    ex.st = stream;
    ex.phase = "bwd";
    ex.pre(tag);
    dp.trace = v.trace;
    dp.trace_id = v.trace_id;
    dp.stats = pl->d_dwa_stats;
    if (const char* knob = getenv("DRVAE_B200_DWA_DEBUG")) dp.debug_flags = atoi(knob);
    cudaError_t r = dwadam_launch(dp, stream, max_ctas);
    ex.post();
    ex.st = keep;
    if (r != cudaSuccess) ex.err = r;
    pl->launches++;
  };
  // Early part of that launch: the decoder heads' tiles as soon as the decoder's dX GEMM (the last reader of their
  // weights) has been enqueued, on dwa_early_sms SMs of a low-priority stream; the persistent GEMMs of the rest of
  // the chain are capped to the other SMs while it runs.
  bool dwa_early_done = false;
  const int nsm = gemm_num_sms();
  const bool dwa_early = ex.defer_dw && !use_stepk && !pl->prof_on &&
                         pl->dwa_early_tiles > 0 && pl->dwa_early_tiles < pl->dwa_tiles && pl->dwa_early_sms >= 8 &&
                         pl->dwa_early_sms <= nsm - 16;

  ex.phase = "";
  cudaStream_t cm = own_main ? pl->s_main : st;
  if (own_main) cudaStreamWaitEvent(cm, pl->ev.begin, 0);
  ex.st = cm;
  auto rows_grid = [&](int rows) { return dim3(cdiv(rows, ROW_WARPS), E); };
  auto row_items = [&](int rows) { return cdiv(rows, STEPK_ROWS); };
  // (While recording for the step kernel the streams only define the levels.)
  const bool overlap = pl->has_fprop && !pl->prof_on;
  cudaStream_t side = overlap ? pl->s_side : cm;
  auto on = [&](cudaStream_t s) { ex.st = s; };
  auto after = [&](cudaStream_t waiter, cudaEvent_t ev, cudaStream_t producer) {
    if (!overlap || waiter == producer) return;
    if (ex.rec) {
      ex.rec->after(waiter, producer);
      return;
    }
    cudaEventRecord(ev, producer);
    cudaStreamWaitEvent(waiter, ev, 0);
  };
  // gradient path (stand-alone weight-gradient GEMMs inside the chain): they run on the plan's main stream, unused
  // there, next to the dX chain on the caller's stream
  const bool dw_aside = backward && !fused_adam && overlap;
  ex.dw_stream = dw_aside ? pl->s_main : nullptr;
  ex.dw_event = pl->ev.dw;
  if (dw_aside && !use_stepk) {
    cudaEventRecord(pl->ev.dw, cm);  // (the split-K path zeroes the gradient buffer on the caller's stream first)
    cudaStreamWaitEvent(pl->s_main, pl->ev.dw, 0);
  }
  auto launch_noise = [&]() {
    const drvae_eps_layout_t& el = pl->epsl;
    EpsSegs sg{};
    const long long offs[6] = {el.off_x1, el.off_x2, el.off_z1, el.off_z2, el.off_z2f, el.off_z3};
    const int outer[6] = {1, 1, L, L, L, L};
    // the input noise (segments 0, 1) is drawn inside prep_kernel with the same keys
    const int inner[6] = {0, 0, pl->Z, pl->has_pair ? pl->Z : 0, pl->has_T ? pl->Z : 0, pl->has_fprop ? pl->Y * pl->Z3 : 0};
    long long most = 0;
    for (int i = 0; i < 6; ++i) {
      sg.off[i] = offs[i];
      sg.outer[i] = outer[i];
      sg.inner[i] = inner[i];
      most = std::max(most, (long long)outer[i] * N * ((inner[i] + 3) / 4));
    }
    dim3 g((unsigned)((most + 255) / 256), E, 6);
    ex.pre("philox_normal");
    launch_k(philox_normal_kernel, g, dim3(256), 0, ex.st, pl->eps_own, sg, N, pl->Ncap, pl->d_dyn, v.trace, v.trace_id);
    ex.chk();
  };
  // step kernel: the noise generator needs only this step's scalars, so it is forked first and overlaps rowmap / prep
  if (use_stepk && own_eps) {
    if (overlap) {
      after(side, pl->ev.noise, cm);
      on(side);
    }
    launch_noise();
    on(cm);
  }
  ex.pre("rowmap");
  launch_k(rowmap_kernel, dim3(E), dim3(ROWMAP_THREADS), 0, cm, v);
  ex.chk();
  ex.pre("prep");
  launch_k(prep_kernel, dim3(round_up(R0b, 128) / PREP_ROWS, cdiv(pl->view.Xc, PREP_SLAB), E), dim3(PREP_THREADS), 0, cm, v);
  ex.chk();
  // latent noise: on the side stream, forked AFTER prep so that it fills the SMs next to the encoder GEMMs instead of
  // running in front of prep (it is first needed by sample_q1)
  if (own_eps && !use_stepk) {
    after(side, pl->ev.noise, cm);  // after this step's scalars (set_dyn), rowmap and prep
    on(side);
    launch_noise();
    on(cm);
  }
  if (use_stepk) {
    if (own_eps) after(cm, pl->ev.eps, side);  // the step kernel starts after the noise generator
    ex.rec = &recorder;
  }

  // ---- encoder q(z1|x1), shared with q(z2|x2) (DrVAE.py:408,418) ----
  ex.phase = "enc.fwd";
  ex.block_hidden_fwd(pl->enc, v.Ain, 0, CNT_R0, R0b);
  ex.gemm_nt(pl->enc.H.back(), 0, pl->enc.head, EPI_STORE_F32,
             ex.epi_f32(v.Q.p, v.Q.ms, 2 * pl->view.Zs, 2 * pl->view.Zs, &pl->enc.head), CNT_R0, R0b);
  if (own_eps && !use_stepk) after(cm, pl->ev.eps, side);  // latent noise of this step
  ex.row_op(SROW_SAMPLE_Q1, "sample_q1", row_items(N + PAD_WARPS), 0, [&]() {
    launch_k(pl->view.Zc <= 128 ? sample_q1_kernel<4> : sample_q1_kernel<MAXJ>, rows_grid(N + PAD_WARPS), dim3(ROW_THREADS), 0, cm, v);
  });
  // The label-dependent branch (q(z_top|z1,y) -> p(z1|z_top,y), forward and backward dX: small GEMMs + row kernels
  // that leave most SMs idle) is independent of the decoder branch: side stream between a fork here and a join
  // before the encoder backward.
  after(side, pl->ev.fork, cm);

  auto fprop_fwd_gemms = [&]() {
    // ---- label-dependent part: q(z_top|z1,y), p(z1|z_top,y) per (row, class) evaluation ----
    ex.phase = "z3.fwd";
    ex.block_hidden_fwd(pl->z3b, v.Z1e, 0, CNT_F, Fb);
    ex.gemm_nt(pl->z3b.H.back(), 0, pl->z3b.head, EPI_STORE_F32,
               ex.epi_f32(v.Q3.p, v.Q3.ms, 2 * pl->view.Z3s, 2 * pl->view.Z3s, &pl->z3b.head), CNT_F, Fb);
    ex.row_op(SROW_Z3_POST, "z3_post", row_items(round_up(Fb, 128)), 0,
              [&]() { launch_k(pl->view.Z3c <= 128 ? z3_post_kernel<4> : z3_post_kernel<MAXJ>, rows_grid(round_up(Fb, 128)), dim3(ROW_THREADS), 0, ex.st, v); });
    ex.phase = "dz1.fwd";
    ex.block_hidden_fwd(pl->dz1b, v.Z3b, 0, CNT_F, Fb);
    ex.gemm_nt(pl->dz1b.H.back(), 0, pl->dz1b.head, EPI_STORE_F32,
               ex.epi_f32(v.PZ1.p, v.PZ1.ms, 2 * pl->view.Zs, 2 * pl->view.Zs, &pl->dz1b.head), CNT_F, Fb);
  };
  // the classifier's input gradient (DZ1, DZ2F): d loss / d logits and, with hidden layers, dPre of the last one
  // (+ its zero padding rows), then their dX (+ dW) GEMMs and the split of d u into DZ1 / DZ2F
  auto clf_back = [&]() {
    ex.phase = "clf.bwd";
    if (pl->clf_nh == 0)
      ex.row_op(SROW_CLF_BACK, "clf_back", row_items(LNb), 0,
                [&]() { launch_k(clf_back_kernel, rows_grid(LNb), dim3(ROW_THREADS), 0, ex.st, v); });
    if (pl->clf_nh > 0) {
      if (pl->act == DRVAE_ACT_SOFTPLUS)
        ex.row_op(SROW_CLF_BACK_H_SP, "clf_back", row_items(round_up(LNb, 128)), 0, [&]() {
          launch_k(clf_back_h_kernel<EPI_DSP_C8>, rows_grid(round_up(LNb, 128)), dim3(ROW_THREADS), 0, ex.st, v);
        });
      else
        ex.row_op(SROW_CLF_BACK_H, "clf_back", row_items(round_up(LNb, 128)), 0, [&]() {
          launch_k(clf_back_h_kernel<EPI_DACT_C8>, rows_grid(round_up(LNb, 128)), dim3(ROW_THREADS), 0, ex.st, v);
        });
      const bool split_du = pl->clf_in > pl->Z;
      float* du = split_du ? pl->clfv.dU.p : v.DZ1.p;
      const long long du_ms = split_du ? pl->clfv.dU.ms : v.DZ1.ms;
      // (their weight gradients stay on this stream: the classifier's gradient bucket is recorded here)
      cudaStream_t keep_dw = ex.dw_stream;
      ex.dw_stream = nullptr;
      ex.block_bwd_hidden(pl->clfb, pl->clfv.U, 0, pl->clf_in, du, du_ms, CNT_LN, LNb);
      ex.dw_stream = keep_dw;
      if (split_du)
        ex.row_op(SROW_CLF_DU, "clf_du", row_items(LNb), 0,
                  [&]() { launch_k(clf_du_kernel, rows_grid(LNb), dim3(ROW_THREADS), 0, ex.st, v); });
    }
  };
  // classifier weight gradient (+ Adam in the fused step): feeds nothing but the optimizer
  auto clf_grad = [&]() {
    ex.phase = "clf.bwd";
    if (pl->clf_nh == 0)
      ex.row_op(SROW_CLF_GRAD_PARTIAL, "clf_grad_partial", v.clf_splits, 0,
                [&]() { launch_k(clf_grad_partial_kernel, dim3(v.clf_splits, E), dim3(256), 0, ex.st, v); });
    else  // linear_p over the last hidden activation
      ex.row_op(SROW_CLF_GRAD_PARTIAL_H, "clf_grad_partial", v.clf_splits, 0,
                [&]() { launch_k(clf_grad_partial_h_kernel, dim3(v.clf_splits, E), dim3(256), 0, ex.st, v); });
    ex.row_op(SROW_CLF_GRAD_REDUCE, "clf_grad_reduce", row_items(pl->Y * (pl->clf_pin + 1)), 0, [&]() {
      launch_k(clf_grad_reduce_kernel, dim3(cdiv(pl->Y * (pl->clf_pin + 1), 8), E), dim3(256), 0, ex.st, v);
    });
  };
  auto clf_bwd = [&]() {
    clf_back();
    clf_grad();
  };
  if (pl->has_fprop) {
    on(side);
    fprop_fwd_gemms();
    on(cm);
  }
  // ---- p(z2|z1) ----
  ex.phase = "T.fwd";
  if (pl->has_T) {
    ex.gemm_nt(v.Zdec, 0, pl->Tsh, EPI_STORE_F32, ex.epi_f32(v.PT.p, v.PT.ms, 2 * pl->view.Zs, 2 * pl->view.Zs, &pl->Tsh), CNT_LN, LNb);
    ex.row_op(SROW_T_POST, "T_post", row_items(N + PAD_WARPS), 0, [&]() {
      launch_k(pl->view.Zc <= 128 ? T_post_kernel<4> : T_post_kernel<MAXJ>, rows_grid(N + PAD_WARPS), dim3(ROW_THREADS), 0, ex.st, v);
    });
  }
  if (pl->has_fprop) {
    // pz1_post weighs unlabeled evaluations by q(y|.), which the classifier (T_post for DrVAE, sample_q1 for VFAE,
    // clf_fwd with hidden layers) produces
    after(side, pl->ev.qy, cm);
    on(side);
    if (pl->clf_nh > 0) {
      ex.phase = "clf.fwd";
      if (pl->clf_in > pl->Z)  // DrVAE: u = [z1 | z2f - z1 | 1] (VFAE reads the z1 rows of Zdec)
        ex.row_op(SROW_CLF_U, "clf_u", row_items(LNb), 0,
                  [&]() { launch_k(clf_u_kernel, rows_grid(LNb), dim3(ROW_THREADS), 0, ex.st, v); });
      ex.block_hidden_fwd(pl->clfb, pl->clfv.U, 0, CNT_LN, LNb);
      ex.row_op(SROW_CLF_FWD, "clf_fwd", row_items(LNb), 0,
                [&]() { launch_k(clf_fwd_kernel, rows_grid(LNb), dim3(ROW_THREADS), 0, ex.st, v); });
    }
    if (pl->side_delay_cycles > 0 && !ex.rec) spin_kernel<<<1, 1, 0, ex.st>>>(pl->side_delay_cycles);
    ex.row_op(SROW_PZ1_POST, "pz1_post", row_items(round_up(Fb, 128)), 0,
              [&]() { launch_k(pl->view.Zc <= 128 ? pz1_post_kernel<4> : pz1_post_kernel<MAXJ>, rows_grid(round_up(Fb, 128)), dim3(ROW_THREADS), 0, ex.st, v); });
    // clf_back (main stream) reads the per-class KL terms pz1_post has just written (kfp_row)
    if (overlap && backward && pl->has_clf) ex.ev_record(pl->ev.kfp, ex.st);
    if (backward) {
      if (dwa_early) ex.cta_cap = nsm - pl->dwa_early_sms;  // (they run next to the early dW+Adam launch)
      ex.phase = "dz1.bwd";
      ex.block_bwd(pl->dz1b, v.dY9, v.Z3b, 0, pl->Z3, v.dZ3.p, v.dZ3.ms, CNT_F, Fb);
      if (!ex.rec) cudaEventRecord(pl->bucket_ev[0], ex.dw_stream ? ex.dw_stream : ex.st);
      ex.row_op(SROW_Z3_BACK, "z3_back", row_items(round_up(Fb, 128)), 0,
                [&]() { launch_k(pl->view.Z3c <= 128 ? z3_back_kernel<4> : z3_back_kernel<MAXJ>, rows_grid(round_up(Fb, 128)), dim3(ROW_THREADS), 0, ex.st, v); });
      ex.phase = "z3.bwd";
      ex.block_bwd(pl->z3b, v.dY7, v.Z1e, 0, pl->Z, v.dZ1e.p, v.dZ1e.ms, CNT_F, Fb);
      if (!ex.rec) cudaEventRecord(pl->bucket_ev[1], ex.dw_stream ? ex.dw_stream : ex.st);
      ex.cta_cap = 0;
      // what q_back needs from this stream; the loss reduction that follows here is joined at the end of the step only
      if (overlap) ex.ev_record(pl->ev.side_bwd, ex.st);
    }
    on(cm);
  }
  // ---- decoder p(x|z) on the stacked rows [z1 | z2 | z2f], fused log-density + gradient ----
  ex.phase = "dec.fwd";
  ex.block_hidden_fwd(pl->dec, v.Zdec, 0, CNT_RD, Rdb);
  {
    EpiParams e = ex.epi_base();
    e.out_c8 = pl->dY5.p;
    e.out_c8_ms = pl->dY5.ms;
    e.out_c8_rcap = pl->dY5.rcap;
    e.bias = pl->derived.p + pl->dec.head.bias_off;
    e.bias_ms = pl->derived.ms;
    e.tgt4 = v.tgt4.p;
    e.tgt_ms = v.tgt4.ms;
    e.tgt_rcap = pl->view.R0cap;
    e.X = pl->X;
    e.Xc = pl->view.Xc;
    e.counts = v.counts.p;
    e.counts_stride = (int)v.counts.ms;
    e.coefs = v.coefs.p;
    e.coefs_stride = (int)v.coefs.ms;
    e.L = L;
    e.part = v.dec_part.p;
    e.part_ms = v.dec_part.ms;
    e.part_rcap = pl->view.Rdcap;
    e.write_dy = backward ? 1 : 0;
    ex.gemm_nt(pl->dec.H.back(), 0, pl->dec.head, EPI_DECLOSS, e, CNT_RD, Rdb);
  }
  // The loss reduction is off the backward's critical path: it runs at the tail of the side stream
  // (after that branch's backward), once the decoder log-density partials of the main stream exist.
  after(side, pl->ev.side_fwd, cm);
  on(side);
  ex.phase = "";
  ex.row_op(SROW_LOSS_PARTIAL, "loss", v.loss_slices, v.loss_slices,
            [&]() { launch_k(loss_partial_kernel, dim3(v.loss_slices, E), dim3(256), 0, ex.st, v); });
  ex.row_op(SROW_LOSS_FINAL, "loss_final", 1, 0, [&]() { launch_k(loss_final_kernel, dim3(E), dim3(32), 0, ex.st, v); });
  if (losses_out && ex.ok() && !ex.rec) {
    // losses buffer per model is padded to 256 B in the arena; the caller's is dense [E][8]
    ex.err = cudaMemcpy2DAsync(losses_out, 8 * sizeof(float), v.losses.p, v.losses.ms * sizeof(float),
                               8 * sizeof(float), E, cudaMemcpyDeviceToDevice, ex.st);
  }
  if (overlap) ex.ev_record(pl->ev.side_end, side);  // everything the side stream does in this step
  on(cm);

  if (backward && ex.ok()) {
    size_t bk = pl->has_fprop ? 2 : 0;  // buckets 0, 1 (decoder_z1, encoder_z3) were recorded by the side branch
    auto bucket_done = [&](bool weight_gemm = true) {
      if (!ex.rec) cudaEventRecord(pl->bucket_ev[bk], (weight_gemm && ex.dw_stream) ? ex.dw_stream : ex.st);
      ++bk;
    };
    ex.phase = "dec.bwd";
    if (dwa_early) {
      ex.after_head_dx = [&]() {
        cudaEventRecord(pl->ev.dwa, cm);
        cudaStreamWaitEvent(pl->s_dwa, pl->ev.dwa, 0);
        launch_dwadam(0, pl->dwa_early_tiles, pl->s_dwa, pl->dwa_early_sms, "dw_adam_early");
        ex.phase = "dec.bwd";
        ex.cta_cap = nsm - pl->dwa_early_sms;
        dwa_early_done = true;
      };
    }
    ex.block_bwd(pl->dec, pl->dY5, v.Zdec, 0, pl->Z, v.dZdec.p, v.dZdec.ms, CNT_RD, Rdb);
    bucket_done();
    if (pl->has_clf) {
      if (overlap && pl->has_fprop) ex.ev_wait(cm, pl->ev.kfp);
      if (own_main) {
        // only the input gradient (clf_back) is on the chain towards T_back / q_back; the weight gradient runs on
        // the caller's stream, which is otherwise idle until the main chain joins it in front of the dW+Adam launch
        clf_back();
        after(st, pl->ev.clf, cm);
        on(st);
        clf_grad();
        bucket_done(false);
        on(cm);
      } else {
        clf_bwd();
        bucket_done(false);
      }
    }
    if (pl->has_T) {
      ex.phase = "T.bwd";
      ex.row_op(SROW_T_BACK, "T_back", row_items(N + PAD_WARPS), 0,
                [&]() { launch_k(pl->view.Zc <= 128 ? T_back_kernel<4> : T_back_kernel<MAXJ>, rows_grid(N + PAD_WARPS), dim3(ROW_THREADS), 0, ex.st, v); });
      ex.gemm_dx(v.dYT, pl->Tsh, EPI_STORE_F32, ex.epi_f32(v.dZ1T.p, v.dZ1T.ms, pl->Z, pl->Z, nullptr), CNT_LN, LNb);
      ex.gemm_dw(v.dYT, v.Zdec, 0, pl->Tsh, CNT_LN, LNb);
      bucket_done();
    }
    if (overlap) ex.ev_wait(cm, pl->ev.side_bwd);  // join: q_back sums the side branch's gradients into q(z1|x1)
    ex.phase = "enc.bwd";
    ex.row_op(SROW_Q_BACK, "q_back", row_items(N + PAD_WARPS), 0,
              [&]() { launch_k(pl->view.Zc <= 128 ? q_back_kernel<4> : q_back_kernel<MAXJ>, rows_grid(N + PAD_WARPS), dim3(ROW_THREADS), 0, ex.st, v); });
    ex.block_bwd(pl->enc, v.dY2, v.Ain, 0, pl->X, nullptr, 0, CNT_R0, R0b);
    bucket_done();
  }
  ex.cta_cap = 0;
  if (overlap) ex.ev_wait(cm, pl->ev.side_end);
  if (ex.dw_stream) {  // join the weight-gradient stream
    if (ex.rec) {
      ex.rec->after(cm, ex.dw_stream);
    } else {
      cudaEventRecord(pl->ev.dw_end, ex.dw_stream);
      cudaStreamWaitEvent(cm, pl->ev.dw_end, 0);
    }
  }
  if (ex.rec && ex.ok()) {
    // ---- the recorded chain as one cooperative launch ----
    ex.rec = nullptr;
    ex.st = cm;
    ex.phase = "step";
    StepParams* sp = new StepParams();
    std::vector<std::string> tags;
    int max_items = 1;
    cudaError_t ferr = recorder.finalize(*sp, tags, max_items);
    if (ferr == cudaErrorNotSupported) {
      // more ops than the kernel's tables hold (very deep blocks): this plan keeps the launch-per-kernel schedule.
      // What has been issued so far (noise, rowmap, prep) is idempotent, so the sequence is simply enqueued again.
      delete sp;
      cudaGetLastError();
      pl->stepk_unsupported = true;
      return run_step(pl, b, nz, hp, losses_out, st, backward, fused_adam);
    }
    if (ferr != cudaSuccess) {
      delete sp;
      return set_cuda_error("drvae step kernel tables", ferr);
    }
    sp->t.v = v;
    sp->t.v.trace = nullptr;
    sp->bar = pl->d_stepk_bar;
    sp->dbg = pl->dbg;
    sp->trace = nullptr;
    sp->trace_id0 = 0;
    prof_pre(pl, cm, "step:chain");
    if (pl->trace_on && pl->trace_next + sp->t.n_levels <= pl->trace_cap) {
      sp->trace = pl->d_trace;
      sp->trace_id0 = pl->trace_next;
      pl->trace_next += sp->t.n_levels;
      for (int l = 0; l < sp->t.n_levels; ++l) pl->trace_tags.push_back("L" + std::to_string(l) + "|" + tags[l]);
    }
    cudaError_t lerr = step_kernel_launch(*sp, max_items, cm);
    delete sp;
    prof_post(pl, cm);
    if (lerr != cudaSuccess) ex.err = lerr;
    pl->launches++;
    pl->stepk_launches++;
    if (losses_out && ex.ok()) {
      ex.err = cudaMemcpy2DAsync(losses_out, 8 * sizeof(float), v.losses.p, v.losses.ms * sizeof(float),
                                 8 * sizeof(float), E, cudaMemcpyDeviceToDevice, cm);
    }
    if (backward)
      for (auto& ev : pl->bucket_ev) cudaEventRecord(ev, cm);  // every gradient bucket is complete when the kernel ends
  }
  if (own_main) {  // join the main chain into the caller's stream
    cudaEventRecord(pl->ev.end, cm);
    cudaStreamWaitEvent(st, pl->ev.end, 0);
  }
  ex.st = st;
  if (ex.defer_dw && ex.ok()) {
    if (dwa_early_done) {  // the early part runs on its own stream: the rest starts when both are complete
      cudaEventRecord(pl->ev.dwa_end, pl->s_dwa);
      cudaStreamWaitEvent(st, pl->ev.dwa_end, 0);
    }
    ex.st = st;
    launch_dwadam(dwa_early_done ? pl->dwa_early_tiles : 0, pl->dwa_tiles, st, 0, dwa_early_done ? "dw_adam_rest" : "dw_adam_all");
  }
  if (!ex.ok()) return set_cuda_error("drvae step launch", ex.err);
  return 0;
}

}  // namespace

namespace {

enum { SEQ_TRAIN = 0, SEQ_LOSS = 1, SEQ_GRAD = 2, SEQ_DP = 3 };

// data-parallel optimizer over peer memory (dp_peer.cuh): cross-GPU barrier (tag from the per-step scalars), then ONE
// kernel that sums every rank's gradient and loss shares in rank order and applies Adam; global losses -> losses_out
int run_dp_adam(drvae_plan* pl, float* losses_out, cudaStream_t st) {
  prof_pre(pl, st, "opt:dp_barrier");
  dp_barrier_kernel<<<1, 32, 0, st>>>(pl->dp, pl->d_dyn, pl->dbg);
  prof_post(pl, st);
  AdamArgs a{};
  a.params = MBuf<float>{pl->params, pl->P};
  a.grads = MBuf<float>{pl->grads, pl->P};
  a.m = MBuf<float>{pl->adam_m, pl->P};
  a.v = MBuf<float>{pl->adam_v, pl->P};
  a.shadow = pl->shadow;
  a.derived = pl->derived;
  a.segs = pl->d_segs;
  a.nseg = (int)pl->segs.size();
  a.P = pl->P;
  a.update = 1;
  a.h = &pl->d_dyn->s.mem.adam;
  a.skip_lo = a.skip_hi = 0;
  if (pl->arch.kind == DRVAE_KIND_PVAE && pl->has_T) a.skip_lo = (int)pl->T_range[0], a.skip_hi = (int)(pl->T_range[0] + pl->T_range[1]);
  a.dyn = pl->d_dyn;
  a.counts = pl->view.counts.p;
  a.counts_stride = (int)pl->view.counts.ms;
  const int nred = pl->P + 8;
  prof_pre(pl, st, "opt:adam_peer");
  adam_peer_kernel<<<cdiv(nred, 1024), 256, 0, st>>>(a, pl->dp, nred, losses_out);
  prof_post(pl, st);
  pl->launches += 2;
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) return set_cuda_error("adam_peer_kernel", err);
  if (pl->wn) {
    WnArgs w{pl->d_wn_rows, (int)pl->wn_rows.size(), a.params, a.grads, pl->shadow, pl->derived};
    wn_refresh_kernel<<<dim3(cdiv(w.nrows, 8), pl->E), 256, 0, st>>>(w);
    pl->launches++;
    err = cudaGetLastError();
    if (err != cudaSuccess) return set_cuda_error("wn_refresh_kernel", err);
  }
  pl->shadows_valid = true;
  return 0;
}

// does this train step run the grouped dW+Adam launch (dwadam.cuh) instead of gradient + stand-alone Adam?
bool train_is_fused(const drvae_plan* pl, const drvae_batch_t* b) {
  // Not when build_dwa left it out (weight norm, unbound moments, a layer outside its layout conditions).
  // One (or a few) models on a large minibatch: the weight gradients need split-K to fill the GPU, which the
  // grouped launch does not do (its tiles take the complete sum).  Both -> gradient buffer + stand-alone optimizer.
  if (!pl->dwa_ok) return false;
  if (b && (long long)b->N * pl->L >= 1024 && pl->E < 8) return false;
  return true;
}

// Enqueue the whole launch sequence of one call on `st` (everything after the per-step scalars).
int enqueue_sequence(drvae_plan* pl, int seq, const drvae_batch_t* b, const drvae_noise_t* nz, const drvae_hparams_t* hp,
                     float* losses_out, cudaStream_t st, bool fused) {
  if (seq == SEQ_LOSS) return run_step(pl, b, nz, hp, losses_out, st, false, false);
  if (seq == SEQ_GRAD) {
    int rc = run_step(pl, b, nz, hp, losses_out, st, 2, false);
    if (rc || !pl->wn) return rc;
    rc = run_wn_grad(pl, st);
    // the conversion rewrites every bucket: bucket events must not fire before it
    for (auto& ev : pl->bucket_ev) cudaEventRecord(ev, st);
    return rc;
  }
  if (fused) {
    // forward + ELBO + backward with the weight gradients and Adam of every layer in the grouped launch: no gradient
    // buffer traffic and no separate optimizer pass (the bound gradient buffer is left untouched)
    return run_step(pl, b, nz, hp, losses_out, st, 2, true);
  }
  // split train step and data-parallel step: gradient buffer, weight-norm conversion, stand-alone optimizer.  With
  // peers attached the loss shares go right behind the gradient, where the peer optimizer reduces them with it.
  const bool peers = seq == SEQ_DP && pl->dp_on;
  int rc = run_step(pl, b, nz, hp, peers ? pl->grads + pl->P : losses_out, st, 2, false);
  if (rc) return rc;
  rc = run_wn_grad(pl, st);
  if (rc) return rc;
  return peers ? run_dp_adam(pl, losses_out, st) : run_adam(pl, hp, 1, st);
}

// One call = [set_dyn_kernel(per-step scalars)] + a launch sequence that is identical for every step of the same
// shape and the same buffers.  The second time a (sequence, N, buffers, stream) combination is seen, the sequence is
// captured into a CUDA graph (the side-stream fork/join becomes graph edges); afterwards a step is one graph launch
// with the arguments of the set_dyn node updated.  Not captured: parity runs with a caller-provided eps block,
// drvae_grad_step (its bucket events are consumed outside), profiling passes, and the legacy default stream.
// drvae_dp_train_step is captured whole: its peer barrier and optimizer are plan launches, and no NCCL call is in it.
int step_entry(drvae_plan* pl, int seq, const drvae_batch_t* b, const drvae_noise_t* nz, const drvae_hparams_t* hp,
               float* losses_out, cudaStream_t st) {
  if (!hp) return set_error("drvae: hparams is null");
  if (!b) return set_error("drvae: batch is null");
  // own noise is keyed by the global row row_offset + r in 40 bits (drvae_noise_t): outside [0, 2^40) rows would wrap
  // onto other rows' normals
  if (nz && !nz->eps && (nz->row_offset < 0 || nz->row_offset > DRVAE_MAX_ROWS - (long long)b->N))
    return set_error("drvae: noise.row_offset must be >= 0 and row_offset + N <= 2^40");
  const bool fused = seq == SEQ_TRAIN && train_is_fused(pl, b);
  const StepDyn dyn = make_dyn(nz, hp, fused);
  const bool graphable = pl->graph_enabled && !pl->prof_on && !(nz && nz->eps) && seq != SEQ_GRAD && pl->shadows_valid &&
                         st != nullptr && st != cudaStreamLegacy && st != cudaStreamPerThread;
  if (graphable) {
    std::vector<long long> key = {seq, b->N, (long long)(size_t)b->x1, (long long)(size_t)b->x2, (long long)(size_t)b->y,
                                  (long long)(size_t)b->has_x2, (long long)(size_t)b->has_y, (long long)(size_t)b->row_index,
                                  (long long)b->dataset_rows, (long long)(size_t)losses_out,
                                  (long long)(size_t)st, hp->training, hp->add_noise};
    drvae_plan::GraphEntry& ge = pl->graphs[key];
    ge.last_use = ++pl->graph_clock;
    if (!ge.exec && ge.seen >= 1) {
      // capture (nothing executes during capture)
      const long long l0 = pl->launches;
      cudaError_t err = cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal);
      if (err == cudaSuccess) {
        int rc = push_dyn(pl, dyn, st);
        if (!rc) rc = enqueue_sequence(pl, seq, b, nz, hp, losses_out, st, fused);
        cudaGraph_t graph = nullptr;
        err = cudaStreamEndCapture(st, &graph);
        if (rc || err != cudaSuccess || !graph) {
          if (graph) cudaGraphDestroy(graph);
          cudaGetLastError();
          // this (sequence, shape, buffers) combination is launched kernel by kernel from now on; other combinations
          // may still capture.  The reason is kept for drvae_last_error()-style inspection (drvae_plan_graph_failures).
          ge.seen = -1000000;
          pl->graph_failures++;
          if (rc) return rc;
        } else {
          size_t n = 0;
          cudaGraphGetNodes(graph, nullptr, &n);
          std::vector<cudaGraphNode_t> nodes(n);
          cudaGraphGetNodes(graph, nodes.data(), &n);
          for (size_t i = 0; i < n && !ge.dyn_node; ++i) {
            cudaGraphNodeType ty;
            if (cudaGraphNodeGetType(nodes[i], &ty) != cudaSuccess || ty != cudaGraphNodeTypeKernel) continue;
            cudaKernelNodeParams np{};
            if (cudaGraphKernelNodeGetParams(nodes[i], &np) == cudaSuccess && np.func == (void*)set_dyn_kernel) {
              ge.dyn_node = nodes[i];
              ge.dyn_params = np;
            }
          }
          if (ge.dyn_node && cudaGraphInstantiate(&ge.exec, graph, 0) == cudaSuccess) {
            ge.launches = pl->launches - l0;
            ge.graph = graph;
          } else {
            ge.exec = nullptr;
            ge.seen = -1000000;
            pl->graph_failures++;
            cudaGraphDestroy(graph);
          }
          pl->launches = l0;
        }
      } else {
        cudaGetLastError();
        ge.seen = -1000000;
        pl->graph_failures++;
      }
      if (pl->graphs.size() > 16) {  // bound the cache: drop the least recently used entry
        auto victim = pl->graphs.end();
        for (auto it = pl->graphs.begin(); it != pl->graphs.end(); ++it)
          if (&it->second != &ge && (victim == pl->graphs.end() || it->second.last_use < victim->second.last_use)) victim = it;
        if (victim != pl->graphs.end()) {
          if (victim->second.exec) cudaGraphExecDestroy(victim->second.exec);
          if (victim->second.graph) cudaGraphDestroy(victim->second.graph);
          pl->graphs.erase(victim);
        }
      }
    }
    if (ge.exec) {
      StepDyn value = dyn;
      StepDyn* dst = pl->d_dyn;
      MemberExpand mx = member_expand(pl);
      void* args[3] = {&value, &dst, &mx};
      cudaKernelNodeParams np = ge.dyn_params;
      np.kernelParams = args;
      np.extra = nullptr;
      cudaError_t err = cudaGraphExecKernelNodeSetParams(ge.exec, ge.dyn_node, &np);
      if (err == cudaSuccess) err = cudaGraphLaunch(ge.exec, st);
      if (err != cudaSuccess) return set_cuda_error("drvae: graph replay", err);
      pl->launches += ge.launches;
      pl->graph_replays++;
      return 0;
    }
    ge.seen++;
  }
  int rc = push_dyn(pl, dyn, st);
  if (rc) return rc;
  return enqueue_sequence(pl, seq, b, nz, hp, losses_out, st, fused);
}

}  // namespace

extern "C" int drvae_sync_shadows(drvae_plan_t* pl, void* stream) {
  if (!pl) return set_error("drvae_sync_shadows: null plan");
  drvae_hparams_t hp{};
  return run_adam(pl, &hp, 0, (cudaStream_t)stream);
}

extern "C" int drvae_train_step(drvae_plan_t* pl, const drvae_batch_t* b, const drvae_noise_t* nz, const drvae_hparams_t* hp,
                                float* losses_out, void* stream) {
  if (!pl) return set_error("drvae_train_step: null plan");
  return step_entry(pl, SEQ_TRAIN, b, nz, hp, losses_out, (cudaStream_t)stream);
}

extern "C" int drvae_loss_forward(drvae_plan_t* pl, const drvae_batch_t* b, const drvae_noise_t* nz, const drvae_hparams_t* hp,
                                  float* losses_out, void* stream) {
  if (!pl) return set_error("drvae_loss_forward: null plan");
  return step_entry(pl, SEQ_LOSS, b, nz, hp, losses_out, (cudaStream_t)stream);
}

extern "C" int drvae_grad_step(drvae_plan_t* pl, const drvae_batch_t* b, const drvae_noise_t* nz, const drvae_hparams_t* hp,
                               float* losses_out, void* stream) {
  if (!pl) return set_error("drvae_grad_step: null plan");
  return step_entry(pl, SEQ_GRAD, b, nz, hp, losses_out, (cudaStream_t)stream);
}

extern "C" int drvae_adam_step(drvae_plan_t* pl, const drvae_hparams_t* hp, void* stream) {
  if (!pl || !hp) return set_error("drvae_adam_step: null argument");
  int rc = push_dyn(pl, make_dyn(nullptr, hp, false), (cudaStream_t)stream);
  if (rc) return rc;
  return run_adam(pl, hp, 1, (cudaStream_t)stream);
}

extern "C" int drvae_dp_train_step(drvae_plan_t* pl, const drvae_batch_t* b, const drvae_noise_t* nz, const drvae_hparams_t* hp,
                                   float* losses_out, void* stream) {
  if (!pl || !losses_out) return set_error("drvae_dp_train_step: null argument");
  return step_entry(pl, SEQ_DP, b, nz, hp, losses_out, (cudaStream_t)stream);
}

// ---- data parallelism over NVLink peer memory (dp_peer.cuh) ----
extern "C" int drvae_dp_attach(drvae_plan_t* pl, const drvae_dp_peers_t* peers) {
  if (!pl || !peers) return set_error("drvae_dp_attach: null argument");
  if (pl->E != 1) return set_error("drvae_dp_attach: data-parallel training shards ONE model (ensembles shard by model)");
  if (peers->world < 1 || peers->world > DP_MAX_RANKS || peers->rank < 0 || peers->rank >= peers->world)
    return set_error("drvae_dp_attach: bad rank / world size");
  if (!pl->params || !pl->adam_m || !pl->adam_v) return set_error("drvae_dp_attach: bind parameters and Adam moments first");
  if (pl->member_table) return set_error("drvae_dp_attach: a plan with a member table cannot be data-parallel");
  DpPeers d{};
  d.rank = peers->rank;
  d.world = peers->world;
  for (int r = 0; r < peers->world; ++r) {
    if (!peers->grad_ptrs[r] || !peers->ctl_ptrs[r]) return set_error("drvae_dp_attach: null peer pointer");
    d.grads[r] = peers->grad_ptrs[r];
    d.ctl[r] = peers->ctl_ptrs[r];
  }
  d.grads_mc = peers->grads_multicast;
  pl->dp = d;
  pl->dp_on = true;
  pl->grads = peers->grad_ptrs[peers->rank];  // the gradient kernels write this rank's symmetric vector
  if (!pl->dp_counts) {
    cudaError_t err = cudaMalloc(&pl->dp_counts, 3 * sizeof(long long));
    if (err != cudaSuccess) return set_cuda_error("drvae_dp_attach", err);
  }
  drop_graphs(pl);
  return 0;
}
extern "C" const long long* drvae_dp_counts_ptr(const drvae_plan_t* pl) { return pl ? pl->dp_counts : nullptr; }
extern "C" long long drvae_dp_grad_floats(const drvae_plan_t* pl) { return pl ? (long long)pl->P + 64 : -1; }
extern "C" int drvae_dp_exchange_counts(drvae_plan_t* pl, long long N, long long Np, long long Nlab, long long tag, void* stream) {
  if (!pl || !pl->dp_on) return set_error("drvae_dp_exchange_counts: no peers attached");
  dp_counts_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(pl->dp, N, Np, Nlab, tag, pl->dp_counts, pl->dbg);
  pl->launches++;
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) return set_cuda_error("dp_counts_kernel", err);
  return 0;
}
extern "C" int drvae_set_member_hparams(drvae_plan_t* pl, const drvae_member_hparams_t* members, int count, void* stream) {
  if (!pl) return set_error("drvae_set_member_hparams: null plan");
  if (pl->dp_on) return set_error("drvae_set_member_hparams: a data-parallel plan cannot take a member table");
  if (count == 0 && !members) {
    if (pl->member_table) drop_graphs(pl);  // captured sequences read the table's expansion
    pl->member_table = false;
    return 0;
  }
  if (!members || count != pl->E) return set_error("drvae_set_member_hparams: need n_models entries (or NULL and 0 to clear)");
  for (int k = 0; k < count; ++k) {
    const drvae_member_hparams_t& h = members[k];
    const float nonneg[] = {h.yloss_rate, h.pertloss_rate, h.kl_qz2pz2_rate, h.noise_std, h.lr, h.weight_decay};
    for (float r : nonneg)
      if (!isfinite(r) || r < 0.f)
        return set_error("drvae_set_member_hparams: rates, noise_std, lr and weight_decay must be finite and >= 0");
    for (int j = 0; j < 8; ++j)
      if (!isfinite(h.log_prior_y[j])) return set_error("drvae_set_member_hparams: log_prior_y must be finite");
  }
  cudaError_t err = cudaSuccess;
  if (!pl->d_member_hp) {
    err = cudaMalloc(&pl->d_member_hp, sizeof(drvae_member_hparams_t) * pl->E);
    if (err == cudaSuccess) err = cudaMalloc(&pl->d_member, sizeof(MemberScalars) * pl->E);
    if (err == cudaSuccess) err = cudaMallocHost(&pl->h_member_stage, sizeof(drvae_member_hparams_t) * pl->E);
    if (err == cudaSuccess) err = cudaEventCreateWithFlags(&pl->member_ev, cudaEventDisableTiming);
    if (err != cudaSuccess) return set_cuda_error("drvae_set_member_hparams", err);
  } else {
    err = cudaEventSynchronize(pl->member_ev);  // the previous table may still be on its way out of the staging buffer
    if (err != cudaSuccess) return set_cuda_error("drvae_set_member_hparams", err);
  }
  cudaStream_t st = (cudaStream_t)stream;
  memcpy(pl->h_member_stage, members, sizeof(drvae_member_hparams_t) * pl->E);
  err = cudaMemcpyAsync(pl->d_member_hp, pl->h_member_stage, sizeof(drvae_member_hparams_t) * pl->E, cudaMemcpyHostToDevice, st);
  if (err == cudaSuccess) err = cudaEventRecord(pl->member_ev, st);
  if (err != cudaSuccess) return set_cuda_error("drvae_set_member_hparams", err);
  if (!pl->member_table) drop_graphs(pl);  // the kernels' per-member pointers and strides change
  pl->member_table = true;
  return 0;
}
// Instrumented builds only (-DGEMM_PROFILE_WAITS): copy out (and optionally clear) the per-(mode, epilogue) barrier
// wait counters of gemm.cuh; a normal build reports that the counters are not compiled in.
extern "C" int drvae_debug_wait_stats(unsigned long long* out, int reset) {
#ifdef GEMM_PROFILE_WAITS
  cudaError_t err = cudaDeviceSynchronize();
  if (err == cudaSuccess && out) err = cudaMemcpyFromSymbol(out, g_wait_stats, sizeof(unsigned long long) * 3 * 8 * 8);
  if (err == cudaSuccess && reset) {
    static unsigned long long zeros[3 * 8 * 8];
    err = cudaMemcpyToSymbol(g_wait_stats, zeros, sizeof(zeros));
  }
  if (err != cudaSuccess) return set_cuda_error("drvae_debug_wait_stats", err);
  return 0;
#else
  (void)out;
  (void)reset;
  return set_error("drvae_debug_wait_stats: library built without -DGEMM_PROFILE_WAITS");
#endif
}

extern "C" int drvae_set_graph(drvae_plan_t* pl, int enable) {
  if (!pl) return set_error("drvae_set_graph: null plan");
  pl->graph_enabled = enable != 0;
  if (!enable) drop_graphs(pl);
  return 0;
}
extern "C" long long drvae_plan_graph_replays(const drvae_plan_t* pl) { return pl ? pl->graph_replays : -1; }
extern "C" long long drvae_plan_graph_failures(const drvae_plan_t* pl) { return pl ? pl->graph_failures : -1; }

namespace {

// deterministic mu-path in fp32 from the master parameters (see infer_f32.cuh)
int run_infer_fp32(drvae_plan* pl, const float* x1, int N, const drvae_infer_out_t* out, cudaStream_t st) {
  const int E = pl->E, X = pl->X, Z = pl->Z, Y = pl->Y;
  int maxw = Z;
  for (const MlpBlock* b : {&pl->enc, &pl->dec, &pl->clfb})
    for (int w : b->widths) maxw = std::max(maxw, w);
  if (pl->clf_nh > 0) maxw = std::max(maxw, pl->clf_in);  // u = [z1, z2 - z1] is staged in an activation buffer
  // scratch per model: two activation buffers [N][maxw], z1 / z2 / one spare [N][Z]
  const size_t per = (size_t)pl->Ncap * (2 * (size_t)maxw + 3 * (size_t)Z);
  if (pl->f32ws_floats < per * E) {
    if (pl->f32ws) cudaFree(pl->f32ws);
    pl->f32ws = nullptr;
    cudaError_t err = cudaMalloc(&pl->f32ws, per * E * sizeof(float));
    if (err != cudaSuccess) return set_cuda_error("drvae_infer: fp32 scratch", err);
    pl->f32ws_floats = per * E;
  }
  float* Ha = pl->f32ws;
  float* Hb = Ha + (size_t)pl->Ncap * maxw;
  float* z1s = Hb + (size_t)pl->Ncap * maxw;
  float* z2s = z1s + (size_t)pl->Ncap * Z;
  const long long ws_ms = (long long)per;
  cudaError_t lerr = cudaSuccess;
  auto lin = [&](const float* Xp, long long x_ms, int ldx, int w_off, int b_off, int ldw, int nout, int K, float bconst, int act,
                 const float* resid, long long r_ms, int ldr, float* o, long long o_ms, int ldo) {
    LinF32 a{};
    a.X = Xp, a.x_ms = x_ms, a.ldx = ldx;
    a.W = pl->params + w_off, a.b = pl->params + b_off, a.p_ms = pl->P, a.ldw = ldw;
    a.bconst = bconst, a.resid = resid, a.r_ms = r_ms, a.ldr = ldr;
    a.out = o, a.o_ms = o_ms, a.ldo = ldo;
    a.rows = N, a.nout = nout, a.K = K, a.act = act;
    linear_f32_kernel<<<dim3(cdiv(nout, 64), cdiv(N, 64), E), 256, 0, st>>>(a);
    pl->launches++;
    if (lerr == cudaSuccess) lerr = cudaGetLastError();
  };
  // hidden layers of a block: leaves (h, h_ms, h_ld) on the last activation
  const int hidden_act = pl->act == DRVAE_ACT_SOFTPLUS ? ACT_SOFTPLUS : ACT_ELU;
  auto hidden = [&](const MlpBlock& b, const float* in, long long in_ms, int in_ld, const float*& h, long long& h_ms, int& h_ld) {
    h = in, h_ms = in_ms, h_ld = in_ld;
    for (size_t i = 0; i < b.hidden.size(); ++i) {
      const Shadow& W = b.hidden[i];
      float* dst = (h == Ha) ? Hb : Ha;
      lin(h, h_ms, h_ld, W.w_off[0], W.b_off[0], W.ld, b.widths[i], W.kin, 0.f, hidden_act, nullptr, 0, 0, dst, ws_ms, maxw);
      h = dst, h_ms = ws_ms, h_ld = maxw;
    }
  };
  const long long outZ = (long long)N * Z, outX = (long long)N * X;
  const float* h;
  long long h_ms;
  int h_ld;
  hidden(pl->enc, x1, (long long)N * X, X, h, h_ms, h_ld);
  const Shadow& eh = pl->enc.head;
  float* z1 = out->z1_mu ? out->z1_mu : z1s;
  const long long z1_ms = out->z1_mu ? outZ : ws_ms;
  lin(h, h_ms, h_ld, eh.w_off[0], eh.b_off[0], eh.ld, Z, eh.kin, 0.f, ACT_NONE, nullptr, 0, 0, z1, z1_ms, Z);
  if (out->z1_lv) lin(h, h_ms, h_ld, eh.w_off[1], eh.b_off[1], eh.ld, Z, eh.kin, -2.f, ACT_NONE, nullptr, 0, 0, out->z1_lv, outZ, Z);
  float* z2 = nullptr;
  long long z2_ms = 0;
  if (pl->has_T) {
    const Shadow& T = pl->Tsh;  // blocks.py:349-361: mu = z + z W_mu^T + bias_mu, logvar = lin(z) - 2
    z2 = out->z2_mu ? out->z2_mu : z2s;
    z2_ms = out->z2_mu ? outZ : ws_ms;
    lin(z1, z1_ms, Z, T.w_off[0], T.b_off[0], T.ld, Z, Z, 0.f, ACT_NONE, z1, z1_ms, Z, z2, z2_ms, Z);
    if (out->z2_lv) lin(z1, z1_ms, Z, T.w_off[1], T.b_off[1], T.ld, Z, Z, -2.f, ACT_NONE, nullptr, 0, 0, out->z2_lv, outZ, Z);
  }
  if (pl->has_clf && (out->proba || out->pred)) {
    if (pl->has_T && z2_ms != z1_ms) return set_error("drvae_infer: z1_mu and z2_mu must both be given or both be null");
    ClfF32 c{};
    c.z1 = z1, c.z2 = pl->has_T ? z2 : nullptr, c.z_ms = z1_ms, c.ldz = Z;
    if (pl->clf_nh > 0) {
      // u in fp32 (DrVAE: [z1, z2 - z1] materialised, VFAE: z1 itself), the hidden layers, then linear_p on the last
      const float* u = z1;
      long long u_ms = z1_ms;
      int u_ld = Z;
      if (pl->has_T) {
        clf_u_f32_kernel<<<dim3(cdiv(N * 2 * Z, 256), E), 256, 0, st>>>(z1, z2, z1_ms, Z, N, Ha, ws_ms, maxw);
        pl->launches++;
        if (lerr == cudaSuccess) lerr = cudaGetLastError();
        u = Ha, u_ms = ws_ms, u_ld = maxw;
      }
      hidden(pl->clfb, u, u_ms, u_ld, h, h_ms, h_ld);
      c.z1 = h, c.z2 = nullptr, c.z_ms = h_ms, c.ldz = h_ld;
    }
    c.W = pl->params + pl->clf_w_off, c.b = pl->params + pl->clf_b_off, c.p_ms = pl->P;
    c.ldw = pl->view.clf_ld, c.Y = Y, c.N = N;
    c.Z = pl->clf_nh > 0 ? pl->clf_pin : Z;  // features per input half (DrVAE without hidden layers: z1 and z2 - z1)
    c.proba = out->proba, c.pred = out->pred;
    clf_f32_kernel<<<dim3(cdiv(N, 8), E), 256, 0, st>>>(c);
    pl->launches++;
    if (lerr == cudaSuccess) lerr = cudaGetLastError();
  }
  const Shadow& dh = pl->dec.head;
  for (int half = 0; half < (pl->has_T ? 2 : 1); ++half) {
    float* mu = half == 0 ? out->px1_mu : out->px2_mu;
    float* sg = half == 0 ? out->px1_sg : out->px2_sg;
    if (!mu && !sg) continue;
    hidden(pl->dec, half == 0 ? z1 : z2, half == 0 ? z1_ms : z2_ms, Z, h, h_ms, h_ld);
    if (mu) lin(h, h_ms, h_ld, dh.w_off[0], dh.b_off[0], dh.ld, X, dh.kin, 0.f, ACT_NONE, nullptr, 0, 0, mu, outX, X);
    if (sg) lin(h, h_ms, h_ld, dh.w_off[1], dh.b_off[1], dh.ld, X, dh.kin, 0.f, ACT_SOFTPLUS_EPS, nullptr, 0, 0, sg, outX, X);
  }
  if (lerr != cudaSuccess) return set_cuda_error("drvae_infer (fp32) launch", lerr);
  return 0;
}

}  // namespace

extern "C" int drvae_set_infer_precision(drvae_plan_t* pl, int fp32) {
  if (!pl) return set_error("drvae_set_infer_precision: null plan");
  pl->infer_fp32 = fp32 != 0;
  return 0;
}

extern "C" int drvae_infer(drvae_plan_t* pl, const float* x1, int N, const drvae_infer_out_t* out, void* stream) {
  if (!pl || !x1 || !out) return set_error("drvae_infer: null argument");
  if (!pl->params) return set_error("drvae_infer: plan has no bound parameters");
  if (N < 1 || N > pl->Ncap) return set_error("drvae_infer: N exceeds the plan's max_batch");
  cudaStream_t st = (cudaStream_t)stream;
  if (pl->infer_fp32 && !pl->wn) return run_infer_fp32(pl, x1, N, out, st);
  drvae_hparams_t hp{};
  if (!pl->shadows_valid) {
    int rc = run_adam(pl, &hp, 0, st);
    if (rc) return rc;
  }
  Exec ex;
  ex.pl = pl;
  ex.st = st;
  ex.N = N;
  DevView& v = ex.v;
  v = pl->view;
  v.N = N;
  v.need_grad = 0;
  v.x1 = MBuf<const float>{x1, (long long)N * pl->X};
  v.eps_x1 = MBuf<const float>{pl->eps_own.p, pl->eps_own.ms};  // never read (training = 0)
  v.eps_x2 = v.eps_x1;
  v.params = MBuf<float>{pl->params, pl->P};
  v.clf_w = pl->wn ? MBuf<const float>{pl->derived.p + pl->clf_eff_off, pl->derived.ms}
                   : MBuf<const float>{pl->params + pl->clf_w_off, pl->P};
  v.dyn = pl->d_dyn;
  v.mem = member_base(pl);
  v.mem_stride = pl->member_table ? 1 : 0;
  v.own_noise = 0;
  {
    drvae_hparams_t ihp{};  // eval mode: training = 0, add_noise = 0
    ihp.beta1 = 0.9f, ihp.beta2 = 0.999f;
    int rc = push_dyn(pl, make_dyn(nullptr, &ihp, false), st);
    if (rc) return rc;
  }
  const int E = pl->E;
  const int rows_dec = pl->has_T ? 2 * N : N;
  InferView o{out->z1_mu, out->z1_lv, out->z2_mu, out->z2_lv, out->proba, out->pred};
  auto rows_grid = [&](int rows) { return dim3(cdiv(rows, ROW_WARPS), E); };
  ex.pre("infer_counts");
  infer_counts_kernel<<<E, 128, 0, st>>>(v, rows_dec);
  ex.chk();
  ex.pre("prep");
  prep_kernel<<<dim3(round_up(N, 128) / PREP_ROWS, cdiv(pl->view.Xc, PREP_SLAB), E), PREP_THREADS, 0, st>>>(v);
  ex.chk();
  ex.block_hidden_fwd(pl->enc, v.Ain, 0, CNT_R0, N);
  ex.gemm_nt(pl->enc.H.back(), 0, pl->enc.head, EPI_STORE_F32, ex.epi_f32(v.Q.p, v.Q.ms, 2 * pl->view.Zs, 2 * pl->view.Zs, &pl->enc.head),
             CNT_R0, N);
  ex.pre("infer_z1");
  infer_z1_kernel<<<rows_grid(N + PAD_WARPS), ROW_THREADS, 0, st>>>(v, o, rows_dec);
  ex.chk();
  if (pl->has_T) {
    ex.gemm_nt(v.Zdec, 0, pl->Tsh, EPI_STORE_F32, ex.epi_f32(v.PT.p, v.PT.ms, 2 * pl->view.Zs, 2 * pl->view.Zs, &pl->Tsh), CNT_LN, N);
    ex.pre("infer_z2");
    infer_z2_kernel<<<rows_grid(N), ROW_THREADS, 0, st>>>(v, o);
    ex.chk();
  }
  if (pl->clf_nh > 0 && (out->proba || out->pred)) {
    // classifier hidden layers over u (written by infer_z2 / the z1 rows of Zdec), then the logits row kernel
    ex.block_hidden_fwd(pl->clfb, pl->clfv.U, 0, CNT_LN, N);
    ex.pre("infer_clf");
    clf_h_infer_kernel<<<rows_grid(N), ROW_THREADS, 0, st>>>(v, o);
    ex.chk();
  }
  if (out->px1_mu || out->px2_mu) {
    ex.block_hidden_fwd(pl->dec, v.Zdec, 0, CNT_RD, rows_dec);
    for (int half = 0; half < (pl->has_T ? 2 : 1); ++half) {
      float* mu = half == 0 ? out->px1_mu : out->px2_mu;
      float* sg = half == 0 ? out->px1_sg : out->px2_sg;
      if (!mu || !sg) continue;
      EpiParams e = ex.epi_base();
      e.out_f32 = mu;
      e.out2_f32 = sg;
      e.out_f32_ms = (long long)N * pl->X;
      e.out_ld = pl->X;
      e.bias = pl->derived.p + pl->dec.head.bias_off;
      e.bias_ms = pl->derived.ms;
      e.X = pl->X;
      ex.gemm_nt(pl->dec.H.back(), half * N, pl->dec.head, EPI_DECOUT, e, CNT_N, N);
    }
  }
  if (!ex.ok()) return set_cuda_error("drvae_infer launch", ex.err);
  return 0;
}

// Wait-cycle counters of the grouped dW+Adam kernel's roles (summed over CTAs and launches since the last reset):
// out[8] = epilogue waits for the accumulator / for a state stage, loader waits for a free stage, storer waits for an
// updated stage / for the TMA unit to read it, operand producer waits for a free slot, MMA waits for operands,
// total CTA cycles.  enable != 0 switches the counters on (drops captured graphs), 0 reads them and switches off.
extern "C" int drvae_debug_dwa_stats(drvae_plan_t* pl, int enable, unsigned long long* out) {
  if (!pl) return set_error("drvae_debug_dwa_stats: null plan");
  cudaError_t err = cudaDeviceSynchronize();
  if (enable) {
    if (!pl->d_dwa_stats && err == cudaSuccess) err = cudaMalloc(&pl->d_dwa_stats, 8 * sizeof(unsigned long long));
    if (err == cudaSuccess) err = cudaMemset(pl->d_dwa_stats, 0, 8 * sizeof(unsigned long long));
  } else if (pl->d_dwa_stats) {
    if (out && err == cudaSuccess) err = cudaMemcpy(out, pl->d_dwa_stats, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost);
    cudaFree(pl->d_dwa_stats);
    pl->d_dwa_stats = nullptr;
  }
  drop_graphs(pl);
  if (err != cudaSuccess) return set_cuda_error("drvae_debug_dwa_stats", err);
  return 0;
}

// ---- kernel trace: what really ran when (first CTA start / last CTA end of every launch, %globaltimer) ----
extern "C" int drvae_trace_begin(drvae_plan_t* pl, int max_launches) {
  if (!pl || max_launches < 1) return set_error("drvae_trace_begin: bad argument");
  if (pl->d_trace) cudaFree(pl->d_trace);
  std::vector<unsigned long long> init(2 * (size_t)max_launches);
  for (int i = 0; i < max_launches; ++i) init[2 * i] = ~0ULL, init[2 * i + 1] = 0ULL;
  cudaError_t err = cudaMalloc(&pl->d_trace, sizeof(unsigned long long) * init.size());
  if (err == cudaSuccess) err = cudaMemcpy(pl->d_trace, init.data(), sizeof(unsigned long long) * init.size(), cudaMemcpyHostToDevice);
  if (err != cudaSuccess) return set_cuda_error("drvae_trace_begin", err);
  pl->trace_cap = max_launches;
  pl->trace_next = 0;
  pl->trace_tags.clear();
  pl->trace_on = true;
  pl->trace_saved_graph = pl->graph_enabled;  // slots are per launch: replayed graphs would reuse them
  pl->graph_enabled = false;
  return 0;
}
// out: lines "index tag start_ns end_ns" (nanoseconds of the GPU's global timer)
extern "C" int drvae_trace_end(drvae_plan_t* pl, char* out, int cap) {
  if (!pl || !pl->trace_on) return set_error("drvae_trace_end: no trace in progress");
  pl->trace_on = false;
  pl->graph_enabled = pl->trace_saved_graph;
  cudaError_t err = cudaDeviceSynchronize();
  std::vector<unsigned long long> h(2 * (size_t)pl->trace_next);
  if (err == cudaSuccess && !h.empty())
    err = cudaMemcpy(h.data(), pl->d_trace, sizeof(unsigned long long) * h.size(), cudaMemcpyDeviceToHost);
  cudaFree(pl->d_trace);
  pl->d_trace = nullptr;
  if (err != cudaSuccess) return set_cuda_error("drvae_trace_end", err);
  std::string txt;
  char line[320];
  for (int i = 0; i < pl->trace_next; ++i) {
    snprintf(line, sizeof(line), "%d %s %llu %llu\n", i, pl->trace_tags[i].c_str(), h[2 * i], h[2 * i + 1]);
    txt += line;
  }
  if (out && cap > 0) {
    strncpy(out, txt.c_str(), cap - 1);
    out[cap - 1] = 0;
  }
  return 0;
}

// ---- optional per-launch timing: events around every launch of the plan, accumulated by tag ----
extern "C" int drvae_profile_begin(drvae_plan_t* pl) {
  if (!pl) return set_error("drvae_profile_begin: null plan");
  pl->prof_on = true;
  pl->prof_used = 0;
  pl->prof_tags.clear();
  pl->prof_acc.clear();
  return 0;
}
extern "C" int drvae_profile_end(drvae_plan_t* pl, char* out, int cap) {
  if (!pl) return set_error("drvae_profile_end: null plan");
  pl->prof_on = false;
  cudaError_t err = cudaDeviceSynchronize();
  if (err != cudaSuccess) return set_cuda_error("drvae_profile_end", err);
  for (size_t i = 0; i < pl->prof_tags.size(); ++i) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, pl->prof_ev[2 * i], pl->prof_ev[2 * i + 1]);
    auto& a = pl->prof_acc[pl->prof_tags[i]];
    a.first += 1;
    a.second += ms;
  }
  std::string txt;
  char line[256];
  for (auto& kv : pl->prof_acc) {
    snprintf(line, sizeof(line), "%s %lld %.6f\n", kv.first.c_str(), kv.second.first, kv.second.second);
    txt += line;
  }
  if (out && cap > 0) {
    strncpy(out, txt.c_str(), cap - 1);
    out[cap - 1] = 0;
  }
  pl->prof_used = 0;
  pl->prof_tags.clear();
  return 0;
}
