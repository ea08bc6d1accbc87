/*
 * mcpilco_b200.h — C ABI of libmcpilco_b200.so: the B200 (sm_100a) implementation of MC-PILCO's
 * Monte-Carlo GP particle-rollout hot path (SURVEY.md §8).
 *
 * The reference (merlresearch/MC-PILCO) is pure Python/PyTorch and has no FFI layer; its boundary for
 * this path is the Python class API.  The host-side mirror of that API lives in mc-pilco_b200/ and
 * binds these symbols with ctypes (see INTEGRATION.md).  Each entry point cites the reference
 * function(s) it replaces as file:line relative to the reference root.
 *
 * Conventions
 *   - plain C: PODs, raw DEVICE pointers (unless a parameter says "host"), explicit sizes/strides;
 *   - all matrices are row-major float64; nothing is allocated or freed by the library: outputs and
 *     workspaces are caller-owned (PyTorch's caching allocator in the shipped host layer);
 *   - `stream` is a cudaStream_t passed as void*; every call only enqueues work on it;
 *   - return value 0 = ok, <0 = error (MCP_E_*); mcpilco_last_error() gives the message.  Numerical
 *     failure (non-SPD K, negative variance -> NaN) is NOT an error: NaN propagates to the cost exactly
 *     as in the reference (policy_learning/MC_PILCO.py:451,497).
 *   - there is no CPU fallback: without a CUDA device every compute entry point returns MCP_E_CUDA.
 */
#ifndef MCPILCO_B200_H
#define MCPILCO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MCP_ABI_VERSION 7

#define MCP_MAX_D 32    /* gp-input dimension            */
#define MCP_MAX_DS 16   /* state dimension               */
#define MCP_MAX_DU 8    /* input dimension               */
#define MCP_MAX_E 16    /* number of GPs (outputs)       */
#define MCP_MAX_DP 32   /* policy feature dimension      */
#define MCP_MAX_POLY 3  /* MPK terms of a Volterra sum   */
#define MCP_MAX_DEG 3   /* degree of one MPK term        */

#define MCP_OK 0
#define MCP_E_ARG (-1)     /* bad shape / unsupported configuration */
#define MCP_E_CUDA (-2)    /* CUDA runtime error (no device, launch failure) */
#define MCP_E_WORKSPACE (-3)

/* ---- kernel hyper-parameters of ONE GP, already mapped out of log-space --------------------------
 * k(x,x') = has_se * lambda * exp(-sum_j ((x_j-x'_j) * inv_ls[j])^2)
 *         + sum_{p<n_poly} prod_{f<poly_deg[p]} ( sum_j poly_w2[p][f][j] x_j x'_j + poly_w2[p][f][MCP_MAX_D] )
 * (gpr_lib/GP_prior/Stationary_GP.py:162-170, Sparse_GP.py:426-441,613-646,671-737, GP_prior.py:314-347).
 * inv_ls[j] = 0 / poly_w2[..][j] = 0 encode dimensions outside `active_dims`.
 * sigma_n2 = exp(sigma_n_log)^2 + sigma_n_num^2 (GP_prior.py:87-89), mean0 = constant prior mean. */
typedef struct McpGpSpec {
  int32_t D;
  int32_t has_se;
  int32_t n_poly;
  int32_t poly_deg[MCP_MAX_POLY];
  double lambda;
  double mean0;
  double sigma_n2;
  double inv_ls[MCP_MAX_D];
  double poly_w2[MCP_MAX_POLY][MCP_MAX_DEG][MCP_MAX_D + 1];
} McpGpSpec;

/* ---- one fitted GP: what Model_learning keeps in gp_inputs_tr_list / alpha_list / K_X_inv_list
 * (model_learning/Model_learning.py:163-208) ------------------------------------------------------- */
typedef struct McpGp {
  McpGpSpec spec;
  int32_t N;           /* training points of this output (differs per GP in SoD mode) */
  int32_t ld_kinv;     /* leading dimension of Kinv (>= N) */
  const double* Xtr;   /* [N, D]   */
  const double* alpha; /* [N]      */
  const double* Kinv;  /* [N, ld_kinv] symmetric */
  double var_scale;    /* norm_list[i]**2, Model_learning.py:220-221 */
  /* OPT-IN error-compensated INT8 tensor-core contraction (mcpilco_ozaki_prepare); ozaki_slices == 0 selects the native FP64 path */
  const int8_t* kinv_planes; /* reversed digit planes of Kinv, mcpilco_ozaki_plane_bytes(N, slices) bytes */
  const int32_t* kinv_exp;   /* [N] row exponents */
  int32_t ozaki_slices;      /* 0 (off), 7 (56-bit) or 8 (64-bit operands) */
  int32_t ld_linv;           /* leading dimension of Linv (>= N, even) */
  /* OPTIONAL triangular factor L^-1 (lower, K + sigma_n2 I = L L^T) from mcpilco_gp_precompute: forward-only predicts / rollouts
   * (no Jacobians) then form  w = K* L^-T  over the triangle only and  var = k** - |w|^2 : half the flops of K* Kinv.  NULL = not
   * available (e.g. Kinv came from a log file): the full product is used. */
  const double* Linv;        /* [N, ld_linv] or NULL */
  /* max_n k(x_n, x_n) over the training inputs (INT8 variant only; 0 = unknown): with it the K* kernel bounds a row by
   * |k(x, x_n)| <= sqrt(k(x,x) kdiag_max) and emits the row's digit planes itself instead of a second pass over K* */
  double kdiag_max;
} McpGp;

/* ---- state -> gp-input map and integration (Model_learning.py:450-456,471-493,564-579,670-718) ---- */
typedef struct McpModel {
  int32_t Ds, Du, E, D;
  int32_t kind;     /* 0: delta-state x' = x + d ; 1: speed-integration */
  int32_t use_trig; /* 1: [x[not_angle], sin x[angle], cos x[angle], u] ; 0: [x, u] */
  int32_t n_na, n_a;
  int32_t na_idx[MCP_MAX_DS];
  int32_t a_idx[MCP_MAX_DS];
  int32_t vel_idx[MCP_MAX_E];
  int32_t pos_idx[MCP_MAX_E];
  int32_t particle_pred; /* 0: use the mean only (MC_PILCO.rollout, :368) */
  int32_t _pad;
  double T;
} McpModel;

/* ---- Sum_of_gaussians policies (policy_learning/Policy.py:153-265,268-335,338-403) ---------------- */
typedef struct McpPolicy {
  int32_t kind; /* 0 plain, 1 with_angles [x_na, cos, sin], 2 with_target_trajectory [x, target_t - x] */
  int32_t nb, Dp, Du, Ds;
  int32_t n_na, n_a;
  int32_t na_idx[MCP_MAX_DS];
  int32_t a_idx[MCP_MAX_DS];
  int32_t squash;   /* flg_squash */
  int32_t has_bias;
  int32_t use_drop; /* flg_drop */
  double u_max[MCP_MAX_DU];
  double inv_scale[MCP_MAX_DP]; /* 1/scale_factor */
  const double* log_ls;         /* [Dp]      log_lengthscales   */
  const double* centers;        /* [nb, Dp]  centers            */
  const double* W;              /* [Du, nb]  f_linear.weight    */
  const double* bias;           /* [Du] or NULL                 */
  const double* target_traj;    /* [>=H, Ds] or NULL            */
} McpPolicy;

/* ---- fused cost (policy_learning/Cost_function.py:25-36,53-63,80-101,124-147,170-182) ------------ */
typedef struct McpCost {
  int32_t kind; /* 0 none (caller differentiates states), 1 cart_pole, 2 saturated trajectory,
                   3 saturated distance to target, 4 distance to target */
  int32_t n_idx;
  int32_t idx[MCP_MAX_DS];   /* cart_pole: {angle_index, pos_index}; others: active state dims */
  double target[MCP_MAX_DS]; /* cart_pole: {theta*, p*}; 3/4: target per active dim */
  double inv_ls[MCP_MAX_DS]; /* 1/lengthscale per active dim */
  const double* target_traj; /* kind 2: [>=H, Ds] */
} McpCost;

/* ---- MC_PILCO4PMS measurement model (policy_learning/MC_PILCO.py:846-906) ------------------------ */
typedef struct McpMeas {
  int32_t enabled;
  int32_t n_pos;
  int32_t pos_idx[MCP_MAX_E];
  int32_t vel_idx[MCP_MAX_E];
  double std_pos[MCP_MAX_E];
  double b0, b1, a0, a1; /* scipy.signal.butter(1, fc) */
  double T;
} McpMeas;

/* ---- noise: injected tensors (parity mode) or counter-based Philox4x32-10 (production) ------------
 * Draw order being replaced: Normal.rsample (Model_learning.py:704-705), F.dropout (Policy.py:225,261),
 * torch.randn (MC_PILCO.py:884).  Philox counters are keyed by the GLOBAL particle id so results do
 * not depend on how particles are sharded over GPUs. */
typedef struct McpNoise {
  const double* eps;      /* [H-1, M, E] or NULL -> Philox */
  const uint8_t* masks;   /* [H, M, nb] {0,1} or NULL -> Philox (ignored when p_dropout == 0) */
  const double* meas_eps; /* [H-1, M, n_pos] or NULL -> Philox */
  uint64_t seed;
  uint64_t particle_offset; /* global id of local particle 0 */
  double p_dropout;
  /* optional DEVICE uint64 added to `seed` when the kernels run (wrapping): lets a CUDA graph that was captured once draw fresh
   * noise on every replay — the host bumps the device word, the baked kernel arguments stay (SURVEY.md 8 f1).  NULL = not used. */
  const uint64_t* seed_dev;
} McpNoise;

/* ---- one rollout (MC_PILCO.apply_policy, policy_learning/MC_PILCO.py:615-674 / :808-906) ---------- */
typedef struct McpRollout {
  int32_t M, H;
  int32_t need_grad; /* 1: keep per-step Jacobian checkpoints for mcpilco_rollout_bwd */
  int32_t M_global;  /* particle count of the whole (possibly sharded) rollout, 0 = M.  Kernel mappings are chosen from it so that a
                        shard performs bit-for-bit the arithmetic the unsharded rollout performs on the same particles */
  McpModel model;
  McpPolicy policy;
  McpCost cost;
  McpMeas meas;
  McpNoise noise;
  const McpGp* gps;    /* HOST array of E descriptors (device pointers inside) */
  const double* x0;    /* [M, Ds] initial particles */
  double* states;      /* out [H, M, Ds] */
  double* inputs;      /* out [H, M, Du] */
  double* jac;         /* out [H-1, M, E, D]  d(delta_e)/d(gp-input_d) incl. the sampling term (need_grad) */
  double* pol_in;      /* out [H, M, Ds] state seen by the policy (== states unless meas.enabled); may be NULL
                          when !meas.enabled */
  double* costs;       /* out [H, M] per-particle cost (cost.kind != 0) or NULL */
  double* cost_out;    /* out [2]: {sum_t mean_m c, sum_t std_m c} (cost.kind != 0) or NULL */
  double* cost_stats;  /* out [H, 2]: per step {mean_m c, sum_m (c - mean)^2} for merging across GPUs, or NULL */
  void* workspace;     /* >= mcpilco_rollout_workspace_bytes() */
  size_t workspace_bytes;
} McpRollout;

typedef struct McpRolloutGrad {
  const double* grad_states; /* [H, M, Ds] dL/dstates or NULL; ADDS to the fused cost's gradient when grad_cost != 0 */
  const double* grad_inputs; /* [H, M, Du] or NULL */
  double grad_cost;          /* upstream gradient of the fused expected cost (0 when the loss does not use it) */
  double* g_log_ls;          /* out [Dp]     */
  double* g_centers;         /* out [nb, Dp] */
  double* g_W;               /* out [Du, nb] */
  double* g_bias;            /* out [Du] or NULL */
  double* g_x0;              /* out [M, Ds] or NULL */
} McpRolloutGrad;

int mcpilco_abi_version(void);
const char* mcpilco_last_error(void);
int mcpilco_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* make `device` current for this library's CUDA runtime (call with torch's current device index) */
int mcpilco_set_device(int device);

/* K = k(X1, X2) (+ sigma_n2 I when add_noise and X2 == NULL); X2 == NULL means X2 = X1.
 * Replaces Sum_Independent_GP.get_covariance / RBF.get_covariance / MPK_GP.get_covariance
 * (GP_prior.py:314-335, Stationary_GP.py:162-170, Sparse_GP.py:625-646).  `spec` is a HOST pointer. */
int mcpilco_gp_covariance(const McpGpSpec* spec, const double* X1, int n1, const double* X2, int n2, int add_noise,
                          double* K, int ldk, void* stream);

/* diag k(x,x) without noise.  Replaces get_diag_covariance (GP_prior.py:337-347, Stationary_GP.py:172-181,
 * Sparse_GP.py:443-453,657-668). */
int mcpilco_gp_diag_covariance(const McpGpSpec* spec, const double* X, int n, double* diag, void* stream);

/* Per-model-update precompute: K = k(X,X) + sigma_n2 I, blocked Cholesky K = L L^T, R = L^-1,
 * Kinv = R^T R, alpha = Kinv (y - mean0).  Replaces GP_prior.forward / get_alpha (GP_prior.py:91-115,130-135)
 * as driven by Model_learning.pretrain_gp (Model_learning.py:163-208).  Lfac / Linv (optional, [N, ld], lower triangular with
 * zeros above the diagonal) receive L and R = L^-1. */
size_t mcpilco_gp_precompute_workspace_bytes(int N);
int mcpilco_gp_precompute(const McpGpSpec* spec, const double* Xtr, const double* y, int N, double* alpha,
                          double* Kinv, int ld, double* Lfac, double* Linv, void* workspace, size_t workspace_bytes, void* stream);

/* Greedy subset-of-data selection (GP_prior.get_SOD, gpr_lib/GP_prior/GP_prior.py:232-257): candidates are visited in `order`
 * (DEVICE int array [N], NULL = 0..N-1; order[0] seeds the subset); a candidate joins when the predictive standard deviation of the
 * GP fitted on the current subset exceeds `threshold` at it.  idx_out [N] receives the selected indices, *count_out their number
 * (both DEVICE).  One incremental Cholesky factor instead of a refit per candidate; no host synchronisation inside. */
size_t mcpilco_gp_sod_workspace_bytes(int N);
int mcpilco_gp_sod_select(const McpGpSpec* spec, const double* X, int N, const int* order, double threshold, int* idx_out, int* count_out,
                          void* workspace, size_t workspace_bytes, void* stream);

/* Training objective of the GP hyper-parameters and its analytic gradient:
 *   out[0] = 0.5 ((y - m)^T K^-1 (y - m) + log det K)   (Marginal_log_likelihood.forward, gpr_lib/Likelihood/Gaussian_likelihood.py:12-24,
 *   evaluated on GP_prior.forward's outputs, GP_prior.py:91-115; the reference obtains the gradient by autograd through
 *   torch.cholesky / torch.inverse inside GP_prior.fit_model, GP_prior.py:179-230),
 *   out[1] = d/d lambda, out[2] = d/d mean0, out[3] = d/d sigma_n2, out[4 + j] = d/d inv_ls[j] (j < MCP_MAX_D),
 *   out[4 + MCP_MAX_D + (p * MCP_MAX_DEG + f) * (MCP_MAX_D + 1) + j] = d/d poly_w2[p][f][j].
 * Gradients are with respect to the McpGpSpec fields; the caller applies the chain rule of its parametrisation.
 * `out` is a DEVICE array of mcpilco_gp_nlml_grad_size() doubles. */
int mcpilco_gp_nlml_grad_size(void);
size_t mcpilco_gp_nlml_workspace_bytes(int N);
int mcpilco_gp_nlml(const McpGpSpec* spec, const double* X, const double* y, int N, double* out, void* workspace,
                    size_t workspace_bytes, void* stream);

/* Posterior at M test inputs for E GPs: mean[m,e] = mean0 + K* alpha, var[m,e] = var_scale (k** - k*^T Kinv k*),
 * and (optional) their Jacobians w.r.t. the test input, jmean/jvar [M, E, D].
 * Replaces GP_prior.get_estimate_from_alpha (GP_prior.py:137-155) as called by
 * Model_learning.get_exact_gp_estimate / get_SOD_gp_estimate (Model_learning.py:265-289,315-336).
 * `gps` is a HOST array. */
size_t mcpilco_gp_predict_workspace_bytes(int M, int Nmax);
int mcpilco_gp_predict(const McpGp* gps, int E, const double* Xs, int M, double* mean, double* var, double* jmean,
                       double* jvar, void* workspace, size_t workspace_bytes, void* stream);

/* Particle rollout forward (MC_PILCO.apply_policy / MC_PILCO4PMS.apply_policy, MC_PILCO.py:615-674,808-906;
 * get_next_state Model_learning.py:210-229; policies Policy.py:242-265; fused Expected_cost) and the
 * hand-written backprop-through-time that replaces cost.backward() (MC_PILCO.py:522). */
size_t mcpilco_rollout_workspace_bytes(int M, int H, int E, int D, int Nmax, int nb, int Dp, int Du);
int mcpilco_rollout_fwd(const McpRollout* r, void* stream);
int mcpilco_rollout_bwd(const McpRollout* r, const McpRolloutGrad* g, void* stream);

/* u[M, Du] = pi(x[M, Ds]) at time index t: sum of Gaussians, dropout (injected masks for step t or Philox), linear layer,
 * tanh squashing.  Replaces Sum_of_gaussians.forward and its two wrappers (policy_learning/Policy.py:242-265,323-335,
 * 389-403).  `masks_t` is [M, nb] or NULL. */
int mcpilco_policy_forward(const McpPolicy* policy, int M, int t, const double* x, double p_dropout, const uint8_t* masks_t,
                           uint64_t seed, uint64_t particle_offset, double* u, void* stream);

/* Vector-Jacobian product of mcpilco_policy_forward: given g_u[M, Du] = dL/du, writes dL/dx [M, Ds] (g_x may be NULL) and
 * dL/d{log_ls [Dp], centers [nb, Dp], W [Du, nb], bias [Du] (NULL if !has_bias)}.  The arguments mean what they mean for the
 * forward, including the dropout mask (the same injected masks_t, or the same Philox draws for (seed, particle_offset + m, t, b)).
 * Outputs are overwritten, not accumulated; M == 0 writes zeros.  Sums over particles are reduced in a fixed order: repeated
 * calls on one device are bit-identical.  `workspace` holds mcpilco_policy_backward_workspace_bytes(M, nb, Dp, Du) bytes. */
size_t mcpilco_policy_backward_workspace_bytes(int M, int nb, int Dp, int Du);
int mcpilco_policy_backward(const McpPolicy* policy, int M, int t, const double* x, double p_dropout, const uint8_t* masks_t,
                            uint64_t seed, uint64_t particle_offset, const double* g_u, double* g_x, double* g_log_ls,
                            double* g_centers, double* g_W, double* g_bias, void* workspace, size_t workspace_bytes, void* stream);

/* Initial particles (MC_PILCO.apply_policy, policy_learning/MC_PILCO.py:635-657) from counter-based Philox keyed by the
 * global particle id:  kind 0: x0 = a[k] + b[k] * n, n ~ N(0, I)  (a = mean, b = sqrt(var); n_modes > 1 draws the mode k
 * uniformly per particle: the multi-modal Gaussian of :640-647);  kind 1: x0 = a + (b - a) * u, u ~ U(0,1) (a = low, b = up
 * bound, :635-639).  a, b are DEVICE arrays [n_modes, Ds]; seed_dev as in McpNoise (NULL = unused). */
int mcpilco_init_particles(int kind, const double* a, const double* b, int n_modes, int M, int Ds, uint64_t seed,
                           uint64_t particle_offset, const uint64_t* seed_dev, double* x0, void* stream);

/* Timing hook for bench.py's roofline: when enabled, every launch of the dominant kernel (the FP64 tensor-core GEMM
 * V = K* Kinv of the posterior) is bracketed by CUDA events on the launching stream.  read() synchronises those events and
 * returns the summed kernel time (ms), the number of bracketed launches and their summed flop count (2 m n k each). */
int mcpilco_prof_enable(int on);
int mcpilco_prof_read(double* total_ms, uint64_t* launches, double* flops);

/* OPT-IN variant of the posterior contraction V = K* Kinv on the INT8 tensor cores (tcgen05) with error compensation (Ozaki scheme:
 * `slices` balanced base-256 digit planes per operand, exact int32 plane products, fp64 recombination).  slices = 8 reproduces the
 * fp64 contraction to ~1e-12 relative, slices = 7 to ~1e-9 (tolerances on the posterior variance: DESIGN.md).  prepare() slices one
 * GP's Kinv once per model update into caller-owned buffers that are then referenced from McpGp.  The contraction index is cut into
 * segments of at most 65536 / slices columns (exact int32 accumulation), recombined in fp64. */
int mcpilco_ozaki_available(void);
size_t mcpilco_ozaki_plane_bytes(int N, int slices);
int mcpilco_ozaki_prepare(const double* Kinv, int N, int ld, int slices, int8_t* planes, int32_t* exponents, void* stream);
/* the contraction on its own: V[M, N] (ldv) = A[M, N] (lda) * Kinv^T from Kinv's prepared planes (used by mcpilco_gp_predict /
 * mcpilco_rollout_fwd when McpGp.ozaki_slices != 0; exported for tests and benchmarks) */
size_t mcpilco_ozaki_scratch_bytes(int M, int N, int slices);
int mcpilco_ozaki_contract(const double* A, int lda, int M, int N, int slices, const int8_t* planes, const int32_t* exponents, double* V,
                           int ldv, void* scratch, size_t scratch_bytes, void* stream);

/* sizeof() of {McpGpSpec, McpGp, McpModel, McpPolicy, McpCost, McpMeas, McpNoise, McpRollout, McpRolloutGrad};
 * returns how many there are.  Lets a binding check its struct layout. */
int mcpilco_struct_sizes(size_t* out, int n);

/* number of kernels this library launched since the last reset (bench.py's gpu_launches) */
uint64_t mcpilco_launch_count(int reset);

#ifdef __cplusplus
}
#endif
#endif /* MCPILCO_B200_H */
