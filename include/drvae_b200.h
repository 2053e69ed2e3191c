/* drvae_b200 — C ABI of the B200-native (sm_100a) DrVAE / PertVAE / VFAE training step.
 *
 * This is the drop-in boundary of SURVEY.md §8(b).  The reference (rampasek/DrVAE) has no FFI:
 * its seam is Python method dispatch on the model object, so each entry point below names the
 * reference method it replaces (paths relative to /root/reference/src):
 *
 *   drvae_train_step    DGMMixin.py:91-126  run_on_batch(train_mode=True): zero_grad,
 *                       loss_function (DrVAE.py:545, PVAE.py:411, VFAE.py:403), backward, Adam.step
 *   drvae_loss_forward  DGMMixin.py:110-115 run_on_batch(train_mode=False): eval-mode losses
 *   drvae_grad_step     the forward+backward half of run_on_batch (for data-parallel runs: the
 *   + drvae_adam_step   caller all-reduces the flat gradient between the two calls)
 *   drvae_infer         DrVAE.py:253-311 / PVAE.py:206-246 / VFAE.py:178-215  forward()
 *   drvae_sync_shadows  after load_state_dict (DGMMixin.py:199-203) or any external write to params
 *
 * Conventions
 *   - plain C, no torch types; every pointer is a DEVICE pointer unless stated otherwise
 *   - status return: 0 = ok, non-zero = error, text from drvae_last_error() (thread local);
 *     nothing throws or aborts; there is no CPU fallback
 *   - ownership: the caller (PyTorch) owns parameters, Adam moments, gradients, batches and
 *     outputs; the plan owns only its workspace and the bf16 weight shadows
 *   - all work is enqueued on the caller's stream; calls are asynchronous
 *   - an "ensemble" is n_models identically shaped, independent models trained in one launch
 *     sequence (grouped GEMMs); every per-model array is laid out [n_models][...]
 */
#ifndef DRVAE_B200_H
#define DRVAE_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define DRVAE_KIND_DRVAE 0
#define DRVAE_KIND_PVAE 1
#define DRVAE_KIND_VFAE 2
#define DRVAE_MAX_HIDDEN 4
#define DRVAE_MAX_CLF_WIDTH 4096
#define DRVAE_MAX_L 256                 /* Monte-Carlo samples per row (drvae_arch_t.L) */
#define DRVAE_MAX_MODELS (1 << 20)      /* n_models of one plan */
#define DRVAE_MAX_ROWS (1LL << 40)      /* global rows addressable by own noise (drvae_noise_t.row_offset + N) */

typedef struct drvae_plan drvae_plan_t;

/* Architecture = constructor arguments of the reference classes that shape tensors
 * (DrVAE.py:45-70, PVAE.py:45-63, VFAE.py:42-60) with the run_*.py fixed choices:
 * type_rec='diag_gaussian', nonlinearity='elu', type_y='discrete', clf_z1z2=True,
 * use_s=False, use_MMD=False, dropout 0, batch norm off.  The classifier's hidden layers (dim_h_clf, --class-y)
 * are an argument of drvae_plan_create_clf; drvae_plan_create builds the classifier without them. */
typedef struct {
  int kind;                /* DRVAE_KIND_* */
  int dim_x, dim_y;
  int dim_z1;
  int dim_z3;              /* DrVAE dim_z3 / VFAE dim_z2 (top latent); ignored for PVAE */
  int n_enc_z1, enc_z1[DRVAE_MAX_HIDDEN];   /* --enc-z1 */
  int n_dec_x, dec_x[DRVAE_MAX_HIDDEN];     /* --dec-x  */
  int n_enc_z3, enc_z3[DRVAE_MAX_HIDDEN];   /* --enc-z3 (DrVAE) / --enc-z2 (VFAE) */
  int n_dec_z1, dec_z1[DRVAE_MAX_HIDDEN];   /* --dec-z1 */
  int weight_norm;         /* layers.WeightNormLinear instead of nn.Linear (model.wn) */
  int L;                   /* --L: Monte-Carlo samples per row */
  int max_batch;           /* row capacity per model (--batch-size) */
} drvae_arch_t;

/* One minibatch per model, reference layout (DrVAE.py:956-961): x1, x2 float32 [n_models][N][dim_x]
 * row-major; y, has_x2, has_y int32 [n_models][N].  Unused fields may be NULL (x2/has_x2 for
 * VFAE, y/has_y for PVAE).  s is not consumed (use_s=False).  Zero-initialise the struct: optional fields added
 * at its end must be NULL / 0 when unused. */
typedef struct {
  const float* x1;
  const float* x2;
  const int* y;
  const int* has_x2;
  const int* has_y;
  int N;
  /* Device-resident dataset (the reference's fit() draws minibatches from an in-memory dataset through a sampler,
   * src/DrVAE.py:743-781, src/utils.py:292-327): when row_index is non-NULL the arrays above hold dataset_rows rows per
   * model and the minibatch is rows row_index[model][0..N) of them (int32, device).  The step reads the dataset
   * through the indices; nothing is gathered or copied.  NULL: the arrays are the minibatch itself. */
  const int* row_index;
  int dataset_rows;
} drvae_batch_t;

/* Noise.  eps != NULL: parity mode, a row-indexed block of standard normals per model laid out
 * as drvae_eps_layout() reports.  eps == NULL: the step draws its own with Philox4x32-10 keyed by
 * (seed, step, model, draw kind, MC sample, row_offset + row, feature): a data-parallel shard that
 * passes the global index of its first row draws the noise of the unsharded minibatch.  The counter holds the
 * model in 20 bits, the MC sample in 8 and the global row in 40, so every key is distinct only inside these ranges,
 * which the library enforces: n_models <= 2^20 and L <= 256 (drvae_plan_create), and with eps == NULL
 * 0 <= row_offset and row_offset + N <= 2^40 (each step entry point). */
typedef struct {
  const float* eps;
  unsigned long long seed;
  long long row_offset;
} drvae_noise_t;

/* Scalars of one step (reference: DrVAE.py:79-97 internals, run_drvae.py:173-185 ctor call). */
typedef struct {
  int step;               /* finished_training_iters before this step (Adam t = step + 1) */
  int training;           /* 1: train mode (input noise if add_noise), 0: eval mode */
  int add_noise;          /* --train-w-noise */
  float noise_std;        /* --noise-var, used as a std multiplier (DrVAE.py:406) */
  float beta_pert;        /* _compute_anneal_coef(step, itermax, offset), DGMMixin.py:77-89 */
  float pertloss_rate, kl_qz2pz2_rate, yloss_rate;
  float kl_min;           /* free bits, 2.0 */
  float lr, beta1, beta2, adam_eps, weight_decay;
  int global_N, global_Np, global_Nlab;  /* >0: batch-global normalisers (data-parallel shards) */
  float log_prior_y[8];   /* log prior over classes ('uniform' -> log(1/dim_y)) */
  /* optional: DEVICE pointer to {N, Np, Nlab} as int64, already summed over the shards (e.g. by an NCCL all-reduce
   * enqueued on the same stream).  Overrides global_* when non-NULL, so a data-parallel step needs no host round
   * trip for its normalisers. */
  const long long* global_counts_dev;
} drvae_hparams_t;

/* Per-member hyperparameters of an ensemble (heterogeneous ensembles: a learning-rate x loss-rate x fold grid in one
 * plan).  With a table set, these fields of member m replace the same fields of drvae_hparams_t for that member;
 * everything else (step, training, add_noise, beta_pert, kl_min, Adam betas and epsilon, global counts) still comes from
 * drvae_hparams_t.  log_prior_y as in drvae_hparams_t. */
typedef struct {
  float yloss_rate, pertloss_rate, kl_qz2pz2_rate;
  float noise_std;
  float lr, weight_decay;
  float log_prior_y[8];
} drvae_member_hparams_t;

/* Layout of the row-indexed eps block (floats, per model; Ncap = max_batch):
 *   x1   [Ncap][dim_x]            input noise of x1 rows
 *   x2   [Ncap][dim_x]            input noise of x2 rows (indexed by the row of the pair)
 *   z1   [L][Ncap][dim_z1]        sample of q(z1|x1)
 *   z2   [L][Ncap][dim_z1]        second sample of q(z1|x1) used as z2 (reference quirk)
 *   z2f  [L][Ncap][dim_z1]        sample of p(z2|z1)
 *   z3   [L][Ncap][dim_y][dim_z3] top latent; slot 0 for a labeled row, slot j for class j */
typedef struct {
  long long off_x1, off_x2, off_z1, off_z2, off_z2f, off_z3, total;
} drvae_eps_layout_t;

/* Outputs of drvae_infer, all [n_models][N][...] device buffers owned by the caller; any may be
 * NULL.  (DrVAE.py:310-311 dictionary.) */
typedef struct {
  float* z1_mu;   float* z1_lv;    /* qz1                       [N][dim_z1] */
  float* z2_mu;   float* z2_lv;    /* pz2 = p(z2|z1=mu)         [N][dim_z1] (DrVAE, PVAE) */
  float* proba;   int* pred;       /* clamp(softmax), argmax    [N][dim_y], [N] (DrVAE, VFAE) */
  float* px1_mu;  float* px1_sg;   /* p(x1|z1)                  [N][dim_x] */
  float* px2_mu;  float* px2_sg;   /* p(x2|z2)                  [N][dim_x] (DrVAE, PVAE) */
} drvae_infer_out_t;

const char* drvae_last_error(void);

int drvae_plan_create(const drvae_arch_t* arch, int n_models, drvae_plan_t** out);
/* The same with n_clf hidden ELU layers of widths clf_hidden[0..n_clf) in front of the classifier's linear_p
 * (CategoricalDecoder = blocks.MLP + linear_p, dim_h_clf / --class-y): n_clf in [0, DRVAE_MAX_HIDDEN], every width in
 * [1, DRVAE_MAX_CLF_WIDTH], n_clf = 0 on a PVAE plan (it has no classifier).  n_clf = 0 is drvae_plan_create.
 * Their tensors come before linear_p: encoder_y.nnet.model.linear{1..n_clf}.{weight, bias[, g]}. */
int drvae_plan_create_clf(const drvae_arch_t* arch, int n_clf, const int* clf_hidden, int n_models, drvae_plan_t** out);
int drvae_plan_destroy(drvae_plan_t* plan);

/* Parameter layout: tensors in the reference's state_dict order (SURVEY.md Appendix C), each row-major at `offset`
 * floats inside the flat per-model vector of drvae_plan_param_count().  Every tensor and every matrix ROW starts on
 * a 16-byte boundary: element (r, c) of tensor i lives at offset + r * drvae_plan_tensor_ld(i) + c, with
 * ld = cols rounded up to a multiple of 4 (1 for vectors).  The padding floats are zero parameters with zero
 * gradients and stay zero; Adam moments and gradients use the same layout. */
long long drvae_plan_param_count(const drvae_plan_t* plan);
int drvae_plan_num_tensors(const drvae_plan_t* plan);
int drvae_plan_tensor_info(const drvae_plan_t* plan, int index, char* name, int name_cap, int* rows, int* cols,
                           long long* offset);
int drvae_plan_tensor_ld(const drvae_plan_t* plan, int index);   /* floats between rows; -1: bad index */
int drvae_plan_eps_layout(const drvae_plan_t* plan, drvae_eps_layout_t* out);
long long drvae_plan_workspace_bytes(const drvae_plan_t* plan);

/* Bind caller-owned state: params, adam_m, adam_v, grads are float32 [n_models][param_count]. */
int drvae_plan_bind(drvae_plan_t* plan, float* params, float* adam_m, float* adam_v, float* grads);
int drvae_sync_shadows(drvae_plan_t* plan, void* stream);

/* losses_out: float32 [n_models][8] = RECL, KLD, PERT, YL, MMD, ELBO, CMPL, 0 (device). */
int drvae_train_step(drvae_plan_t* plan, const drvae_batch_t* batch, const drvae_noise_t* noise,
                     const drvae_hparams_t* hp, float* losses_out, void* stream);
int drvae_loss_forward(drvae_plan_t* plan, const drvae_batch_t* batch, const drvae_noise_t* noise,
                       const drvae_hparams_t* hp, float* losses_out, void* stream);
int drvae_grad_step(drvae_plan_t* plan, const drvae_batch_t* batch, const drvae_noise_t* noise,
                    const drvae_hparams_t* hp, float* losses_out, void* stream);
int drvae_adam_step(drvae_plan_t* plan, const drvae_hparams_t* hp, void* stream);

/* Member table.  members: HOST array of n_models entries, or NULL with count 0 to clear the table.  Stream-ordered:
 * the table is copied to the plan's device copy on `stream` and takes effect from the next step enqueued on `stream`,
 * including graph replays (replacing one table by another keeps captured graphs; setting or clearing one drops them).
 * Each step expands the table into per-member Adam and loss scalars on the device, so a member's update is
 * bit-identical to that of a table-less plan whose drvae_hparams_t carries the member's values.  Errors: a count other
 * than n_models or 0, a non-finite value, a negative rate, lr or noise_std, and a plan with drvae_dp_attach done
 * (either order: drvae_dp_attach also refuses a plan with a table). */
int drvae_set_member_hparams(drvae_plan_t* plan, const drvae_member_hparams_t* members, int count, void* stream);

/* Gradient buckets for data-parallel overlap.  drvae_grad_step completes the flat gradient in
 * contiguous ranges ("buckets", one per network block, reported here in completion order) and
 * records a CUDA event after each; drvae_stream_wait_bucket makes `stream` wait for bucket i of the
 * most recent drvae_grad_step, so the caller can all-reduce it while backward is still running. */
int drvae_plan_num_buckets(const drvae_plan_t* plan);
int drvae_plan_bucket_info(const drvae_plan_t* plan, int index, long long* offset, long long* count);
int drvae_stream_wait_bucket(drvae_plan_t* plan, int index, void* stream);
/* Data parallelism over NVLink peer memory (one model, rows of the minibatch sharded over the GPUs of one box).
 * Every rank keeps its flat gradient (+ its 8 additive loss shares right behind it: drvae_dp_grad_floats() floats) and
 * a control block of 128 int64 in allocations ALL ranks have mapped; the caller passes the peer pointers
 * (torch.distributed._symmetric_memory, cudaIpc handles, ...).  Per step:
 *   drvae_dp_exchange_counts   batch-global normalisers {N, Np, Nlab}: posted to all peers, summed into
 *                              drvae_dp_counts_ptr() (pass it as drvae_hparams_t.global_counts_dev); also the barrier
 *                              that keeps a fast rank from overwriting a gradient a slow rank still reads
 *   drvae_dp_train_step        forward + backward into the own gradient vector, the loss shares right behind it (they
 *                              join the reduction), then a cross-GPU barrier (tag = step + 1, read from the per-step
 *                              scalars) + ONE kernel that sums every rank's gradient over NVLink in rank order and
 *                              applies Adam and the shadow refresh; global losses -> losses_out (device, 8 floats)
 * grads_multicast (optional): NVLS multicast mapping of the gradient vectors; the sum is then formed inside the
 * switch (multimem.ld_reduce).  No NCCL call is involved; results are bit-identical on all ranks. */
typedef struct {
  int rank, world;
  float* const* grad_ptrs;        /* [world] device pointers to every rank's gradient vector (own rank included) */
  long long* const* ctl_ptrs;     /* [world] device pointers to every rank's control block (zeroed before attach) */
  float* grads_multicast;         /* or NULL */
} drvae_dp_peers_t;
int drvae_dp_attach(drvae_plan_t* plan, const drvae_dp_peers_t* peers);
long long drvae_dp_grad_floats(const drvae_plan_t* plan);
const long long* drvae_dp_counts_ptr(const drvae_plan_t* plan);
int drvae_dp_exchange_counts(drvae_plan_t* plan, long long N, long long Np, long long Nlab, long long tag, void* stream);
/* One data-parallel optimisation step, always through the gradient buffer and the stand-alone optimizer (never the
 * grouped dW+Adam launch of drvae_train_step).  With peers attached: the exchange above.  Without: this rank's rows
 * alone, drvae_grad_step + drvae_adam_step in one call, losses -> losses_out [n_models][8].  Replayed as a CUDA graph
 * like drvae_train_step. */
int drvae_dp_train_step(drvae_plan_t* plan, const drvae_batch_t* batch, const drvae_noise_t* noise,
                        const drvae_hparams_t* hp, float* losses_out, void* stream);
int drvae_infer(drvae_plan_t* plan, const float* x1, int N, const drvae_infer_out_t* out, void* stream);
/* Inference arithmetic.  fp32 != 0 (default): the mu-path is evaluated with fp32 operands and fp32 accumulation from
 * the master parameters, so that class probabilities agree with the reference to ~1e-6 and thresholded predictions
 * match it exactly; 0: the bf16 tensor-core GEMMs of the training step (faster, probabilities within ~1e-3).  Plans
 * with weight norm always use the tensor-core path. */
int drvae_set_infer_precision(drvae_plan_t* plan, int fp32);

/* Reconstruction metrics of the evaluation path: DeepGenerativeModelMixin.eval_x_reconstruction, src/DGMMixin.py:128-158
 * (numpy RMSE, sklearn r2_score(multioutput='variance_weighted'), the Python loop of scipy.stats.pearsonr over rows, the
 * mean per-row Gaussian log-likelihood of src/blocks.py:230-234).  x, x_rec, x_sigma: fp32 [N][X] row-major device
 * buffers (x_sigma may be NULL: ll = NaN); mask: optional int32 [N], rows with mask == 0 are left out (the reference
 * indexes the labeled / paired rows first); out: 4 doubles on the device {rmse, r2, pearr, ll}; workspace: device
 * buffer of drvae_eval_workspace_bytes(N, X) bytes.  fp64 arithmetic like the reference, fixed-order reductions. */
long long drvae_eval_workspace_bytes(int N, int X);
int drvae_eval_x_reconstruction(const float* x, const float* x_rec, const float* x_sigma, const int* mask, int N, int X,
                                double* out, void* workspace, void* stream);

/* Every metric of the evaluation path for E models (ensemble members) in one call: the reconstruction metrics above
 * for x1 and x2, and the y metrics of DeepGenerativeModelMixin.eval_y_prediction (src/DGMMixin.py:160-190): accuracy,
 * sklearn roc_auc_score and average_precision_score, binary on proba[:, 1] for Y == 2, one-vs-rest with a macro
 * average for Y > 2.  Member m's rows are its D rows with valid != 0; x2 metrics use those with has_x2 != 0 too, y
 * metrics those with has_y != 0 too.  Padding rows (valid == 0) have no effect, whatever they hold.
 *
 * All buffers are [E][D](...) row-major device buffers.  A group left entirely NULL gives NaN in its output columns;
 * px1_sg / px2_sg NULL give ll = NaN.  out: device [E][11] doubles, columns in this fixed order:
 *   0 y_acc, 1 y_auroc, 2 y_aupr, 3 x1_rmse, 4 x1_r2, 5 x1_pearr, 6 x1_ll, 7 x2_rmse, 8 x2_r2, 9 x2_pearr, 10 x2_ll
 * A member without a selected row gets NaN for that group.  auroc / aupr are NaN when a selected row has a label outside
 * [0, Y) or a non-finite score (binary: column 1; Y > 2: any column); a score column whose rows are all of one class
 * gives auroc NaN and ap 1 (all positive) or 0 (none positive), as sklearn 1.9 does.  AUROC and AP are computed from
 * exact integer counts (no sort), fp64 sums in a fixed order: two calls give bit-identical results, and E = 1 with
 * only x1 equals drvae_eval_x_reconstruction bit for bit.  workspace: drvae_eval_members_workspace_bytes(E, D, X, Y)
 * bytes (Y < 2: no y group). */
typedef struct {            /* all [E][D](...) row-major device buffers; a NULL group gives nan in its outputs */
  const int* valid;                                      /* [E][D], required */
  const float* x1; const float* px1_mu; const float* px1_sg;   /* [E][D][X]; px1_sg may be NULL */
  const float* x2; const float* px2_mu; const float* px2_sg;   /* [E][D][X]; NULL for VFAE */
  const int* has_x2;                                     /* [E][D] */
  const float* proba; const int* pred; const int* y; const int* has_y;   /* [E][D][Y], [E][D] x3; NULL for PVAE */
} drvae_eval_members_in_t;
long long drvae_eval_members_workspace_bytes(int E, int D, int X, int Y);
int drvae_eval_members(const drvae_eval_members_in_t* in, int E, int D, int X, int Y,
                       double* out /* device [E][11] */, void* workspace, void* stream);

/* Launch mechanism.  With graphs enabled (default) drvae_train_step / drvae_loss_forward / drvae_dp_train_step
 * replay their launch sequence as a CUDA graph from the second call with the same (N, batch buffers, output buffer,
 * stream) on; per-step scalars live in device memory, so only one kernel node's arguments change between steps.
 * Calls on the legacy default stream, with a caller-provided eps block, or under profiling are launched kernel by
 * kernel, and so is drvae_grad_step.  drvae_plan_launch_count counts the launches of a replayed graph too. */
int drvae_set_graph(drvae_plan_t* plan, int enable);
long long drvae_plan_graph_replays(const drvae_plan_t* plan);
/* Captures that failed (that call shape then runs as plain launches; other shapes still capture): 0 on a healthy plan. */
long long drvae_plan_graph_failures(const drvae_plan_t* plan);
/* Persistent step kernel (default off: measured slower than the captured graph of launches, DESIGN.md §4): the
 * forward + ELBO + input-gradient chain of a step runs as ONE cooperative launch whose dependent stages are separated
 * by grid barriers instead of kernel boundaries; 0 keeps one launch per GEMM / row operation.  Results do not depend
 * on it (bit-identical).  drvae_plan_step_kernel_launches counts the launches of that kernel (0: the plan fell back to
 * the launch-per-operation schedule). */
int drvae_set_step_kernel(drvae_plan_t* plan, int enable);
long long drvae_plan_step_kernel_launches(const drvae_plan_t* plan);

/* Introspection for tests and bench.py */
int drvae_set_gemm_impl(drvae_plan_t* plan, int impl);   /* 0 tcgen05 (default), 1 SIMT validation kernel */
long long drvae_plan_launch_count(const drvae_plan_t* plan); /* kernels launched by this plan so far */
/* Per-launch CUDA-event timing of everything the plan launches between begin and end; `out`
 * receives lines "phase:kernel launches total_ms". */
int drvae_profile_begin(drvae_plan_t* plan);
int drvae_profile_end(drvae_plan_t* plan, char* out, int cap);
/* Kernel trace: between begin and end every kernel the plan launches stamps the GPU's global timer when its first
 * CTA starts and when its last CTA leaves (graphs are off meanwhile: slots are per launch).  `out` receives lines
 * "index phase:kernel start_ns end_ns": the step as it really ran, streams overlapping (tools/trace_step.py). */
int drvae_trace_begin(drvae_plan_t* plan, int max_launches);
int drvae_trace_end(drvae_plan_t* plan, char* out, int cap);
/* Wait-cycle counters of the grouped weight-gradient + Adam kernel's roles: enable != 0 starts counting; enable == 0
 * copies out[8] = {epilogue waits for accumulator, epilogue waits for a state stage, state loader waits for a free
 * stage, storer waits for an updated stage, storer waits for the TMA unit to read it, operand producer waits for a
 * free slot, MMA waits for operands, total CTA cycles} (host memory) and stops. */
int drvae_debug_dwa_stats(drvae_plan_t* plan, int enable, unsigned long long* out);
/* Barrier-wait cycle counters of the GEMM kernel roles, [3 modes][8 epilogues][8 counters]; only in libraries built
 * with -DGEMM_PROFILE_WAITS (tools/wait_profile.py), otherwise an error status. */
int drvae_debug_wait_stats(unsigned long long* out, int reset);
/* Test knob: hold the plan's side stream for `cycles` SM clocks in front of the kernel whose output the main stream
 * consumes next (pz1_post -> clf_back), so that a missing cross-stream dependency produces a wrong result instead of
 * passing by timing luck (tests/test_step_gpu.py::test_side_stream_delay_does_not_change_results).  0 = off. */
int drvae_debug_side_delay(drvae_plan_t* plan, long long cycles);
int drvae_debug_buffer(drvae_plan_t* plan, const char* name, void** ptr, long long* model_stride_bytes,
                       long long* bytes, int* rcap, int* fcap);
int drvae_debug_gemm(int impl, int mode, const void* A, int a_rcap, int a_nchunks, long long a_ms,
                     const void* B, int b_rcap, int b_nchunks, long long b_ms, float* D, int ldd,
                     long long d_ms, int M, int N, int K, int BN, const int* dyn_dev, int ksplit,
                     int desc_variant, int n_models, void* stream);

#ifdef __cplusplus
}
#endif
#endif
