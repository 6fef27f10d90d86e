/*
 * l2o_b200 — C-ABI of the B200-native coordinate-wise LSTM learned-optimizer engine.
 *
 * The reference (VITA-Group/Open-L2O, L2O-DM / L2O-RNNProp) is pure Python/TensorFlow and has no
 * FFI; the seam this library sits behind is the reference's own operator surface.  Each entry point
 * cites the reference code it replaces (DM/ = "Model_Free_L2O/L2O-DM and L2O-RNNProp/"):
 *
 *   l2o_net_create / l2o_net_destroy    networks.factory + StandardDeepLSTM.__init__   DM/networks.py:34-44,157-205
 *   l2o_theta_count / l2o_theta_layout  snt.get_variables_in_module order              DM/networks.py:47-62
 *   l2o_state_floats                    Network.initial_state_for_inputs               DM/networks.py:234-236,273-276
 *   l2o_workspace_bytes                 the loop-carried tensors + TensorArray of the while_loop  DM/meta.py:361-376
 *   l2o_step                            delta, state' = net(g, state)  (one time step) DM/networks.py:207-232,254-271,287-300
 *                                       + RNNProp Adam features                        DM/meta_rnnprop_train.py:383-388
 *                                       + x_next = x + delta                           DM/meta.py:352-353
 *   l2o_unroll_fwd                      the tf.while_loop body x T                     DM/meta.py:338-376
 *                                       imitation unroll                               DM/meta_dm_train.py:463-480
 *   l2o_unroll_bwd                      tf.gradients(loss, theta) through that loop    DM/meta.py:412 (BPTT; SURVEY.md App. B)
 *   l2o_adam_step                       tf.train.AdamOptimizer(lr).minimize            DM/meta.py:411-413
 *   l2o_log_and_sign                    preprocess.LogAndSign                          DM/preprocess.py:52-70
 *   l2o_lasso_grad                      problems.lasso(_fixed) loss + tf.gradients     DM/problems.py:103-175, DM/meta.py:322-329
 *
 * Conventions: every pointer is a DEVICE pointer owned by the caller (PyTorch allocates); no hidden
 * allocation; `stream` is a cudaStream_t passed as void*; every entry returns 0 or a negative
 * L2O_E_* code and never throws; calls are re-entrant per (device, stream).  All tensors fp32 except
 * the accumulators `fx`, `imit_loss`, `dtheta` which are fp64 (order-independent atomics).
 *
 * Layouts (row-major, N = number of coordinates):
 *   state arena  : for layer l (size H_l):  h_l [N][H_l] then c_l [N][H_l], layers concatenated
 *                  == the reference's tuple over layers of (hidden, cell) tensors [N, H_l].
 *   theta        : flat, Sonnet variable order: [input_projection/w [n_in,F], /b [F],]
 *                  lstm_1/w_gates [F+H1,4H1], lstm_1/b_gates [4H1], lstm_2/w_gates [H1+H2,4H2],
 *                  lstm_2/b_gates [4H2], linear/w [top,1], linear/b [1]; gate column order i|j|f|o.
 *   sequences    : [T][N] time-major; RNNProp feature sequences [T][2][N] (m~ then g~).
 *   ckpt         : [T+1] state arenas; slot t = state BEFORE step t; slot T = final state.
 */
#ifndef L2O_B200_H_
#define L2O_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define L2O_OK 0
#define L2O_E_INVALID (-1)      /* bad argument (NULL where required, n<0, T<0 ...) */
#define L2O_E_UNSUPPORTED (-2)  /* net shape / mode not compiled into this build */
#define L2O_E_CUDA (-3)         /* CUDA runtime error (see l2o_last_cuda_error) */
#define L2O_E_NOMEM (-4)

#define L2O_PRE_IDENTITY 0 /* tf.identity            DM/networks.py:188,221 */
#define L2O_PRE_LOGSIGN 1  /* preprocess.LogAndSign  DM/preprocess.py:42-70 */
#define L2O_PRE_FC 2       /* Linear(dim)+ELU        DM/networks.py:180-183,219 */

#define L2O_OPT_NONE 0
#define L2O_OPT_RASTRIGIN_SEP 1  /* f = fscale*sum(0.5(x-a)^2 - alpha*b*cos(2 pi x) + alpha)   DM/problems.py:177-213, A=I */
#define L2O_OPT_QUADRATIC_DIAG 2 /* f = fscale*sum((a*x-b)^2)                                   DM/problems.py:73-101, W diagonal */
#define L2O_OPT_QUADRATIC_BATCH 3 /* f = fscale*sum_b ||W_b x_b - y_b||^2, dense W_b [d,d] per group of d = opt_group
                                     consecutive coordinates; opt_a = W [n/d][d][d], opt_b = y [n]; exact-fp32 engine
                                     (groups exchange x through shared memory)                   DM/problems.py:73-101 */

#define L2O_ENGINE_AUTO 0
#define L2O_ENGINE_FFMA 1   /* exact-fp32 CUDA-core kernels */
#define L2O_ENGINE_TC 2     /* tcgen05 (3xTF32 error-compensated) kernels */

typedef struct l2o_net* l2o_handle;

typedef struct {
  int32_t n_layers;    /* 0, 1 or 2 */
  int32_t hidden[2];   /* LSTM sizes */
  int32_t preprocess;  /* L2O_PRE_* */
  int32_t n_in;        /* 1: net(g, s) ; 2: RNNprop net(m~, g~, s) */
  int32_t fc_dim;      /* L2O_PRE_FC: projection width */
  float logsign_k;     /* L2O_PRE_LOGSIGN */
  float scale;         /* output scale                DM/networks.py:229-232 */
  int32_t tanh_output; /* 1: tanh(linear)*scale       DM/networks.py:229-230 */
} l2o_net_desc;

typedef struct {
  int64_t n;
  const float* theta;
  const float* in0;     /* [n] g (or m~ when n_in==2 and m==NULL) */
  const float* in1;     /* [n] g~ (n_in==2, operator surface) or NULL */
  float* m;             /* [n] in/out Adam first moment: non-NULL selects the fused RNNProp feature mode */
  float* v;             /* [n] in/out */
  float beta1, beta2;
  float p;              /* float(step + t)            DM/meta_rnnprop_train.py:384,386 */
  const float* state_in;/* state arena */
  float* state_out;     /* may alias state_in */
  float* x;             /* optional [n], x += delta */
  float* delta;         /* optional [n] */
  float* feat_out;      /* optional [2][n]: (m~, g~) actually fed to the net (recorded for BPTT) */
  const int32_t* step_ptr; /* optional DEVICE scalar: when non-NULL, p = float(*step_ptr + t_offset) (CUDA-graph friendly) */
  int32_t t_offset;
  int32_t reuse_weights;   /* 1: theta is unchanged since this handle's previous l2o_step / forward launch on this stream:
                              the tensor-core engine skips rebuilding its weight image (one tiny launch per step saved;
                              the caller steps T times per unroll with the same theta).  0 is always safe. */
} l2o_step_args;

typedef struct {
  int64_t n;
  int32_t T;
  const float* theta;
  const float* in_seq;  /* [T][n_in][n] pre-recorded net inputs, or NULL when opt_kind != NONE */
  int32_t opt_kind;     /* L2O_OPT_*: gradient evaluated in-kernel from x */
  const float* opt_a;
  const float* opt_b;
  float opt_alpha;
  float opt_fscale;
  float* x;             /* [n] in/out (required for in-kernel optimizees; optional otherwise) */
  float* state;         /* state arena in/out (S_0 -> S_T) */
  float* ckpt;          /* optional [T+1] arenas: slots 0..T written (slot 0 = S_0 copy) */
  float* m;             /* fused RNNProp feature mode (with opt_kind != NONE or in_seq = raw g [T][n]) */
  float* v;
  float beta1, beta2;
  int32_t step0;        /* p = float(step0 + t)       DM/util.py:59-60 */
  float* g_rec;         /* optional [T+1][n]: raw gradients g_0..g_T (g_T at x_T) for the lambda suffix sums */
  float* feat_rec;      /* optional [T][2][n]: (m~, g~) per step */
  double* fx;           /* optional [T+1]: fx[t] += f(x_t) (in-kernel optimizees) */
  float* delta_seq;     /* optional [T][n] */
  const float* labels;  /* optional [T][n]: imitation targets      DM/meta_dm_train.py:472-475 */
  double* imit_loss;    /* += sum_t 0.5*sum((label-delta)^2)/n_total */
  int64_t n_total;
  int32_t opt_group;    /* L2O_OPT_QUADRATIC_BATCH: coordinates per dense group (1..128, n % opt_group == 0) */
} l2o_unroll_args;

typedef struct {
  int64_t n;
  int32_t T;
  const float* theta;
  const float* in_seq;  /* [T][n_in][n] what the net was fed (g_rec rows 0..T-1, feat_rec, or the imitation inputs) */
  const float* ckpt;    /* [T+1] arenas (slots 0..T-1 read) */
  const float* g_rec;   /* [T+1][n] raw gradients -> dDelta_t = sum_{tau>t} g_tau ; NULL in imitation mode */
  const float* labels;  /* imitation mode: dDelta_t = (delta_t - label_t)/n_total */
  int64_t n_total;
  double* dtheta;       /* [P] += dL/dtheta */
  const float* delta_seq; /* optional [T][n], imitation mode: the deltas l2o_unroll_fwd recorded for this unroll; lets the
                             tensor-core BPTT form dDelta_t without recomputing the output layer (exact-fp32 engine ignores it) */
  float* scratch;       /* optional [T][n][20] floats, fc(20) nets (RNNProp) only: hand-over buffer between the layer-2 and the
                             layer-1 pass of the tensor-core BPTT; NULL keeps such a net on the exact-fp32 engine */
} l2o_bwd_args;

int l2o_net_create(l2o_handle* out, const l2o_net_desc* desc);
void l2o_net_destroy(l2o_handle h);
int l2o_net_set_engine(l2o_handle h, int32_t engine);
int64_t l2o_theta_count(l2o_handle h);
int64_t l2o_state_floats(l2o_handle h); /* per coordinate: 2*sum(H_l) */
/* Caller-owned buffer sizes (bytes) for n coordinates and an unroll of T steps (SURVEY.md 8(b): l2o_workspace_bytes).
 * fwd_bytes: state arena + [T+1] checkpoint arenas + g_rec [T+1][n] + feat_rec [T][2][n] (n_in == 2 only);
 * bwd_bytes: what l2o_unroll_bwd reads of those (ckpt + g_rec/in_seq) + the fp64 dtheta accumulator.
 * The library itself allocates nothing per call (only a per-net weight image of < 100 KB at first tensor-core use). */
int l2o_workspace_bytes(l2o_handle h, int64_t n, int32_t T, size_t* fwd_bytes, size_t* bwd_bytes);

int l2o_step(l2o_handle h, const l2o_step_args* a, void* stream);
int l2o_unroll_fwd(l2o_handle h, const l2o_unroll_args* a, void* stream);
int l2o_unroll_bwd(l2o_handle h, const l2o_bwd_args* a, void* stream);

/* TF-1.14 Adam on theta: k = 1-based step count. */
int l2o_adam_step(float* theta, const double* dtheta, float* m, float* v, int64_t n, int32_t k, float lr,
                  float beta1, float beta2, float eps, void* stream);

/* out [2][n]: row 0 = max(log(|g|+eps)/k, -1), row 1 = clip(g*e^k, -1, 1). */
int l2o_log_and_sign(const float* g, float* out, int64_t n, float k, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Row-wise dense LSTM net with run-time shapes: StandardDeepLSTM with output_size > 1 = the reference's KernelDeepLSTM
 * (DM/networks.py:154-236,303-351).  A convolution kernel [kw,kh,cin,cout] is R = cin*cout rows of K = kw*kh inputs;
 * with the variable flat in its own order, element (k, r) sits at k*R + r.  theta: lstm_1/w_gates [F+H1,4H1], b_gates,
 * lstm_2/..., linear/w [top, n_out], linear/b [n_out] (F = n_in, or 2*n_in interleaved (log, sign) with LogAndSign);
 * state arena per layer: h [R][H] then c [R][H]; sequences [T][n_in][R]; g_rec [T+1][n_out][R].
 *
 *   l2o_dense_create / destroy / theta_count / state_floats   KernelDeepLSTM.__init__            DM/networks.py:311-323
 *   l2o_dense_step        update, state' = net(kernel_gradient, state)  (+ x += update)          DM/networks.py:329-346
 *   l2o_dense_unroll_bwd  tf.gradients through the unroll for this net (SURVEY.md App. B)         DM/meta.py:412 */
typedef struct l2o_dense* l2o_dense_handle;
typedef struct {
  int32_t n_layers;    /* 0, 1 or 2 */
  int32_t hidden[2];   /* <= 32 */
  int32_t n_in;        /* K raw inputs per row (<= 64 with LogAndSign, <= 128 without) */
  int32_t preprocess;  /* L2O_PRE_IDENTITY | L2O_PRE_LOGSIGN */
  float logsign_k;
  int32_t n_out;       /* outputs per row (<= 64) */
  float scale;
  int32_t tanh_output;
} l2o_dense_desc;
typedef struct {
  int64_t rows;
  const float* theta;
  const float* in;       /* [n_in][rows] */
  const float* state_in;
  float* state_out;      /* may alias state_in */
  float* x;              /* optional [n_out][rows]: x += update */
  float* delta;          /* optional [n_out][rows] */
} l2o_dense_step_args;
typedef struct {
  int64_t rows;
  int32_t T;
  const float* theta;
  const float* in_seq;   /* [T][n_in][rows] */
  const float* ckpt;     /* [T+1] state arenas, slot t = state BEFORE step t */
  const float* g_rec;    /* [T+1][n_out][rows]: dUpdate_t = sum_{tau>t} g_tau ; NULL in imitation mode */
  const float* labels;   /* imitation mode [T][n_out][rows] */
  int64_t n_total;
  double* dtheta;        /* [P] += */
} l2o_dense_bwd_args;
int l2o_dense_create(l2o_dense_handle* out, const l2o_dense_desc* desc);
void l2o_dense_destroy(l2o_dense_handle h);
int64_t l2o_dense_theta_count(l2o_dense_handle h);
int64_t l2o_dense_state_floats(l2o_dense_handle h);   /* per ROW: 2*sum(H_l) */
int l2o_dense_step(l2o_dense_handle h, const l2o_dense_step_args* a, void* stream);
int l2o_dense_unroll_bwd(l2o_dense_handle h, const l2o_dense_bwd_args* a, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Fused gradient producers (SURVEY.md 8(f) row 4): f and df/dx of a synthetic optimizee family in ONE launch, replacing
 * the ~15 TF ops + tf.gradients of the reference's graph (DM/problems.py:103-175, DM/meta.py:322-329).
 *
 *   l2o_lasso_grad   problems.lasso / lasso_fixed:  f = mean_b(0.5 ||A_b x_b - y_b||^2 + l1 ||x_b||_1)
 *                    g = dF/dx;  with `scale` (random-scaling trick, DM/meta_dm_train.py:336-338,384-385) the loss is
 *                    evaluated at x (.) scale and g is multiplied by scale. */
typedef struct {
  int32_t batch, m, n;  /* A [batch][m][n], y [batch][m], x [batch][n] (row-major) */
  const float* A;
  const float* y;
  const float* x;
  const float* scale;   /* optional [batch][n] */
  float l1;
  float* g;             /* [batch][n] */
  double* f;            /* optional scalar: += f */
} l2o_lasso_args;
int l2o_lasso_grad(const l2o_lasso_args* a, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * L2O-Scale HierarchicalRNN update step (SURVEY.md 8(f) row 1; BASELINE config #4).
 * SC/ = Model_Free_L2O/L2O-Scale/L2O-Scale-Training/ ; HR = SC/optimizer/hierarchical_rnn.py.
 *
 *   l2o_hrnn_create            HierarchicalRNN.__init__ + _create_slots (one slot set per optimizee tensor)   HR:69-218
 *   l2o_hrnn_init_state        _initialize_state / _initialize_global_state                                    HR:303-350
 *   l2o_hrnn_prepare           (derived quantities of a fresh / restored state: mean log-lr HR:432-442, first-step
 *                               predicate SC/optimizer/utils.py:128-130, per-tensor gate bias HR:561-575)
 *   l2o_hrnn_step              _compute_updates: one optimizer step over all tensors                          HR:353-430
 *
 * The flag set is the one the reference's drivers run (SC/metarun.py:154-225,243): levels [10,20,20], 4 gradient
 * scales, grad products, log mean-squares, relative lr against the problem-wide mean, gradient shortcut, dynamic
 * output scale, learnable decays / RNN init; no attention.  theta: flat fp32 [l2o_hrnn_theta_count()] in TF variable
 * creation order (documented in open_l2o_b200/hierarchical_rnn.py THETA_SPEC).  state: 21 fp32 planes of [N]
 * (N = sum of tensor sizes, tensors contiguous): 0-9 parameter (hidden), 10 scl_decay, 11 inp_decay,
 * 12 log_learning_rate, 13-16 grad_accum1..4, 17-20 ms1..4.  layer: [n_tensors][20]; global: [20].
 * workspace: caller-owned device buffer of l2o_hrnn_workspace_bytes() bytes, 256-byte aligned; it carries the
 * per-tensor reductions from one step to the next, so it belongs to the state (call l2o_hrnn_prepare after writing
 * the state from outside). */
typedef struct l2o_hrnn* l2o_hrnn_handle;
typedef struct {
  const float* theta;
  float* x;         /* [N] optimizee parameters, updated in place (not needed by init_state / prepare) */
  const float* g;   /* [N] gradients */
  float* state;     /* [21][N] */
  float* layer;     /* [n_tensors][20] per-tensor RNN states */
  float* global;    /* [20] global RNN state */
  void* workspace;
  float* update;    /* optional [N]: the applied step (x_old - x_new) */
} l2o_hrnn_args;
int l2o_hrnn_create(l2o_hrnn_handle* out, const int64_t* tensor_sizes, int32_t n_tensors);
void l2o_hrnn_destroy(l2o_hrnn_handle h);
int64_t l2o_hrnn_theta_count(void);
int64_t l2o_hrnn_state_floats(void);           /* 21 per coordinate */
int64_t l2o_hrnn_coords(l2o_hrnn_handle h);    /* N */
int64_t l2o_hrnn_workspace_bytes(l2o_hrnn_handle h);
int l2o_hrnn_init_state(l2o_hrnn_handle h, const l2o_hrnn_args* a, void* stream); /* all planes but log_learning_rate */
int l2o_hrnn_prepare(l2o_hrnn_handle h, const l2o_hrnn_args* a, void* stream);
int l2o_hrnn_step(l2o_hrnn_handle h, const l2o_hrnn_args* a, void* stream);
/* Sharded use (SURVEY.md 8(e): the one path with an exchange per INNER step).  Every rank holds a contiguous slice of
 * every tensor's coordinates (tensor_sizes given to l2o_hrnn_create are the LOCAL counts, 0 allowed) and replicas of
 * layer / global.  l2o_hrnn_set_global_sizes gives the counts the per-tensor and problem-wide means divide by.  Per
 * step: l2o_hrnn_step_local; all-reduce SUM of the n_doubles fp64 values at the start of the workspace and all-reduce
 * MAX of the n_flags int32 values at flags_offset_bytes (l2o_hrnn_reduce_layout); l2o_hrnn_step_finish.  Same for
 * prepare.  l2o_hrnn_step / l2o_hrnn_prepare are exactly local + finish. */
int l2o_hrnn_set_global_sizes(l2o_hrnn_handle h, const int64_t* global_sizes);
int l2o_hrnn_reduce_layout(l2o_hrnn_handle h, int64_t* n_doubles, int64_t* flags_offset_bytes, int64_t* n_flags);
int l2o_hrnn_prepare_local(l2o_hrnn_handle h, const l2o_hrnn_args* a, void* stream);
int l2o_hrnn_prepare_finish(l2o_hrnn_handle h, const l2o_hrnn_args* a, void* stream);
int l2o_hrnn_step_local(l2o_hrnn_handle h, const l2o_hrnn_args* a, void* stream);
int l2o_hrnn_step_finish(l2o_hrnn_handle h, const l2o_hrnn_args* a, void* stream);

/* Meta-training of the HierarchicalRNN (SC/optimizer/trainable_optimizer.py:200-470: BPTT through the unrolled
 * optimizer; the optimizee's gradients are stop_gradient'ed, :332-338).  The per-parameter level — everything that
 * touches N coordinates — is differentiated by l2o_hrnn_coord_bwd; the per-tensor / global GRUs, the 1/RMS(delta)
 * normalisation, the problem-wide mean log-lr and the objective are [n_tensors x 20]-sized and are differentiated by the
 * host (open_l2o_b200/hrnn_train.py builds them as torch autograd around these two entry points).
 *   forward of one step:   write bias0 / zero_flag / mean_log_lr into the workspace (l2o_hrnn_workspace_layout), zero the
 *                          sums, l2o_hrnn_step_local (planes in place, raw update lr*delta and the per-tensor sums in the
 *                          workspace);
 *   backward of that step: l2o_hrnn_coord_bwd with the planes BEFORE the step and the same per-tensor inputs. */
typedef struct {
  const float* theta;
  const float* state_old;    /* [21][N] planes before the step */
  const float* g;            /* [N] */
  const float* bias0;        /* [n_tensors][32]: injected gate bias r(10) | u(10) | c(10) | pad, as the forward step used it */
  const int32_t* zero_flag;  /* [n_tensors][4] */
  const float* mean_log_lr;  /* [1] */
  const float* d_state_new;  /* [21][N] adjoints of the planes after the step */
  const float* d_upd;        /* [N] adjoint of the raw update lr*delta (before the per-tensor 1/RMS) */
  const float* d_sums;       /* [n_tensors][24] adjoints of the per-tensor sums: h'(10) | feat(12) | delta^2 | log-lr' */
  float* d_state_old;        /* [21][N] out */
  double* d_theta;           /* [theta_count] += (the 739 per-parameter-level weights) */
  double* d_bias0;           /* [n_tensors][32] += */
  double* d_mean_log_lr;     /* [1] += */
} l2o_hrnn_bwd_args;
int l2o_hrnn_coord_bwd(l2o_hrnn_handle h, const l2o_hrnn_bwd_args* a, void* stream);
/* byte offsets inside the workspace: [0] sums (fp64 [n_tensors][24]) [1] any_nz (int32 [n_tensors][4]) [2] zero_flag
 * (int32 [n_tensors][4]) [3] bias0 (fp32 [n_tensors][32]) [4] inv_denom (fp32 [n_tensors]) [5] mean_log_lr (fp32 [1])
 * [6] raw update (fp32 [N]) */
int l2o_hrnn_workspace_layout(l2o_hrnn_handle h, int64_t offsets[7]);

/* ---------------------------------------------------------------------------------------------------------------
 * Hand-written update rules: the two nets of the reference's factory that have no trainable variables.  A rule is one
 * descriptor (no handle, nothing allocated); nothing differentiates through it (the optimizee gradient it consumes is
 * stop-gradient'ed, DM/meta.py:322-329), so there is no backward entry point.
 *
 *   l2o_rule_state_floats   Sgd / Adam .initial_state_for_inputs                  DM/networks.py:370-371,415-420
 *   l2o_rule_step           update, state' = net(g, state)  (+ x += update)       DM/networks.py:367-368,393-413, DM/meta.py:352-353
 *   l2o_rule_unroll_fwd     the tf.while_loop body x T with such a net            DM/meta.py:338-376
 *
 * Arithmetic in fp32 with TF's order and roundings (Sgd: -lr*g ; Adam: t' = t+1, m' = b1*m + (1-b1)*g,
 * v' = b2*v + (1-b2)*g^2, update = -lr*(m'/(1-b1^t')) / (sqrt(v'/(1-b2^t')) + eps)).  The hyper-parameters are
 * doubles because the reference's are Python floats: (1 - b) is formed before the rounding to fp32.
 * Adam state arena: [t, pad, pad, pad | m [n] | v [n]] (t is the fp32 step counter, DM/networks.py:404). */
#define L2O_RULE_SGD 0   /* networks.Sgd    DM/networks.py:354-371 */
#define L2O_RULE_ADAM 1  /* networks.Adam   DM/networks.py:374-420 */
typedef struct {
  int32_t kind;           /* L2O_RULE_* */
  double learning_rate;   /* >= 0 */
  double beta1, beta2;    /* Adam: in [0, 1) */
  double epsilon;
} l2o_rule_desc;
typedef struct {
  int64_t n;
  const float* g;         /* [n] */
  const float* state_in;  /* Adam: arena of n coordinates (t read on the device: CUDA-graph friendly) */
  float* state_out;       /* Adam: must not overlap state_in */
  float* x;               /* optional [n]: x += update */
  float* delta;           /* optional [n]: the update */
} l2o_rule_step_args;
typedef struct {
  int64_t n;
  int32_t T;
  int32_t opt_kind;       /* L2O_OPT_RASTRIGIN_SEP | L2O_OPT_QUADRATIC_DIAG (others: L2O_E_UNSUPPORTED) */
  const float* opt_a;
  const float* opt_b;
  float opt_alpha;
  float opt_fscale;
  float* x;               /* [n] in/out: x_0 -> x_T */
  float* state;           /* Adam: arena in/out (S_0 -> S_T) */
  double* fx;             /* optional [T+1]: fx[t] += f(x_t) */
} l2o_rule_unroll_args;
int l2o_rule_state_floats(const l2o_rule_desc* d, int64_t n, int64_t* out); /* Sgd 0, Adam 4 + 2n */
int l2o_rule_step(const l2o_rule_desc* d, const l2o_rule_step_args* a, void* stream);
int l2o_rule_unroll_fwd(const l2o_rule_desc* d, const l2o_rule_unroll_args* a, void* stream);

/* Number of this library's kernels launched so far in this process (bench.py's gpu_launches). */
int64_t l2o_launch_count(void);
const char* l2o_status_string(int status);
const char* l2o_last_cuda_error(void);
const char* l2o_version(void);

#ifdef __cplusplus
}
#endif
#endif /* L2O_B200_H_ */
